#!/usr/bin/env python3
"""bench.py — tracks/s of the per-track analysis hot path on B200 (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # CUDA path (this repo)
    python bench.py --impl reference --gpus N --steps K ...   # the reference algorithm on the host cores
    python bench.py --workload c4|c5 ...                      # BASELINE.json configs[3] / configs[4] instead of configs[1]
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's results as DIR/<name>.npy

A "step" is one pass of analyze_audio over one batch of synthetic tracks.  Default workload C2 = BASELINE.json configs[1]:
1024 three-minute 44.1 kHz tracks per B200 (BPM 70-180, random keys; SURVEY.md §8d).  The batch is generated ON the device
before the timed region, so `value` is the device-resident throughput.  `e2e` is the same metric through the host-buffer
C-ABI call on pinned host samples (H2D of the samples and D2H of the results inside the timed region):

  * `e2e.value`      one process, ONE call of stratum_b200_analyze_batch with device_ids = [0 .. N-1] on N x tracks-per-GPU
                     host tracks — the library's own multi-device path (what replaces the reference's par_iter,
                     examples/analyze_batch.rs:239-326).  Under torchrun rank 0 makes the call after every rank has released
                     its GPU memory; the other ranks wait at a barrier.
  * `e2e.per_rank`   every rank calls stratum_b200_analyze_batch on its own GPU with its own tracks-per-GPU host tracks
                     (N processes, max time over ranks).  At N = 1 the two are the same call.

One process per GPU under torchrun for the device-resident leg; tracks are independent, so ranks share nothing but the barrier
and the max-over-ranks time (weak scaling: the same batch per GPU at every N).

The reference arm times the CPU oracle port of the reference algorithm (the Rust crate cannot be built in this image: no cargo)
with all host threads on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes as C
import datetime
import json
import os
import statistics
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

SR = 44100
N_SAMPLES = 7_938_000  # 3 minutes
FLOPS_KEY_FRAME = 532_480   # 8192-point frame, 5 N log2 N convention (SURVEY.md §8d)
FLOPS_BASE_FRAME = 112_640  # 2048-point frame

WORKLOADS = {
    "c2": ("tracks_per_sec_3min_44k1",
           "C2: batch of synthetic 3-min 44.1 kHz mono tracks, BPM 70-180, random keys (BASELINE.json configs[1]); analyze_audio defaults"),
    "c4": ("tracks_per_sec_60min_mix",
           "C4: single 60-min synthetic DJ mix with tempo drift 120->128 BPM (BASELINE.json configs[3]); analyze_audio defaults; replicas only (one track = one GPU)"),
    "c5": ("tracks_per_sec_ragged_30s_10min",
           "C5: ragged batch of 30 s - 10 min tracks at 44.1/48 kHz, multi-resolution escalation and key detection enabled (BASELINE.json configs[4])"),
}


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.stop_flag, self.th = index, [], threading.Event(), None

    def _run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def start(self):
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()

    def stop(self):
        self.stop_flag.set()
        if self.th:
            self.th.join(timeout=6)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for nm, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def bind_to_gpu_numa(device_index: int) -> str:
    """Pins this process (and the library's upload thread, which inherits the mask) to the CPUs of the NUMA node the GPU hangs
    off, before any pinned host buffer is allocated: pinned pages are placed on the allocating thread's node, and an upload
    that has to cross the socket interconnect runs at about half the PCIe rate.  Returns a short note for the JSON line."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        bus = pynvml.nvmlDeviceGetPciInfo(h).busId
        bus = (bus.decode() if isinstance(bus, bytes) else bus).lower()
        if len(bus.split(":")[0]) == 8:  # NVML prints an 8-digit domain, sysfs a 4-digit one
            bus = bus[4:]
        node = int(Path(f"/sys/bus/pci/devices/{bus}/numa_node").read_text().strip())
        if node < 0:
            return "gpu numa node unknown (-1)"
        cpus = set()
        for part in Path(f"/sys/devices/system/node/node{node}/cpulist").read_text().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = os.sched_getaffinity(0) & cpus
        if not allowed:
            return f"gpu on numa node {node}, none of its cpus in this process's cpuset"
        os.sched_setaffinity(0, allowed)
        return f"bound to numa node {node} ({len(allowed)} cpus) of GPU {device_index}"
    except Exception as e:  # placement is an optimisation, never a reason to fail the measurement
        return f"not bound ({type(e).__name__})"


def c2_param_rows(first: int, count: int) -> np.ndarray:
    import synth

    out = np.zeros((count, 5), np.float32)
    for i in range(count):
        p = synth.c2_params(first + i)
        out[i] = (p.bpm, p.tonic, p.minor, p.phase_frac, p.chord_amp)
    return out


def workload_layout(workload: str, first: int, count: int):
    """(lengths, sample rates, per-track generator parameters, expected BPMs) of `count` tracks starting at global index `first`."""
    import synth

    if workload == "c2":
        rows = c2_param_rows(first, count)
        return np.full(count, N_SAMPLES, np.uint64), np.full(count, SR, np.uint32), rows, rows[:, 0].copy()
    if workload == "c5":
        ps = [synth.c5_params(first + i) for i in range(count)]
        rows = np.array([[p.bpm, p.tonic, p.minor, p.phase_frac, p.chord_amp] for p in ps], np.float32)
        return np.array([p.n_samples for p in ps], np.uint64), np.array([p.sample_rate for p in ps], np.uint32), rows, rows[:, 0].copy()
    if workload == "c4":
        return np.full(count, 158_760_000, np.uint64), np.full(count, SR, np.uint32), None, np.full(count, 124.0, np.float32)
    raise ValueError(workload)


def fill_device(S, torch, workload, buf, offsets, lens, srs, rows, device):
    """Generates the batch on the device (C2, C5) or uploads the host-rendered mix (C4), outside every timed region."""
    import synth

    if workload == "c2":
        S.synth_batch(buf.data_ptr(), len(lens), N_SAMPLES, SR, rows, device)
    elif workload == "c5":
        for i in range(len(lens)):
            S.synth_batch(buf.data_ptr() + 4 * int(offsets[i]), 1, int(lens[i]), int(srs[i]), rows[i:i + 1], device)
    else:
        x = torch.from_numpy(synth.c4_mix())
        for i in range(len(lens)):
            buf[int(offsets[i]):int(offsets[i + 1])].copy_(x)
    torch.cuda.synchronize()


def oracle_batch(samples: np.ndarray, offsets: np.ndarray, srs: np.ndarray, jobs: int) -> float:
    """Wall seconds of the CPU oracle over the given concatenated tracks with `jobs` threads
    (mirrors rayon par_iter over tracks, examples/analyze_batch.rs:239-326)."""
    import oracle_lib as O

    L = O.lib(fast=True)
    n = len(offsets) - 1
    offs = np.ascontiguousarray(offsets, np.uint64)
    srs = np.ascontiguousarray(srs, np.uint32)
    return float(L.so_batch_timed(O.f32ptr(samples), offs.ctypes.data_as(C.POINTER(C.c_uint64)), srs.ctypes.data_as(C.POINTER(C.c_uint32)), n, jobs,
                                  None, None, None))


def host_jobs() -> int:
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 2)
    return max(1, min(n - 1, 32))  # default_jobs = CPUs - 1 (examples/analyze_batch.rs:180-185), capped to bound the sample


def cpu_sample(workload: str, n_tracks: int):
    """Bounded CPU sample of a workload: (samples, offsets, srs, note, units) — units = how many whole tracks the sample stands for."""
    import synth

    if workload == "c2":
        xs = [synth.render(synth.c2_params(i)) for i in range(n_tracks)]
        srs = [SR] * n_tracks
        note, units = f"{n_tracks} C2 tracks (3 min each)", float(n_tracks)
    elif workload == "c5":
        ps = []
        i = 0
        while len(ps) < n_tracks:  # tracks of at most 4 minutes keep the sample bounded; the rate is quoted per second of audio too
            p = synth.c5_params(i)
            if p.n_samples / p.sample_rate <= 240:
                ps.append(p)
            i += 1
        xs = [synth.render(p) for p in ps]
        srs = [p.sample_rate for p in ps]
        note, units = f"{n_tracks} C5 tracks of <= 4 min", float(n_tracks)
    else:
        n = 6 * 60 * SR  # the first 6 minutes of the mix per worker; a whole mix is ten times that
        x = synth.c4_mix(n)
        xs = [x] * n_tracks
        srs = [SR] * n_tracks
        note, units = f"{n_tracks} x the first 6 minutes of the C4 mix (value scaled by 1/10 to whole 60-min mixes)", n_tracks / 10.0
    offsets = np.zeros(len(xs) + 1, np.uint64)
    offsets[1:] = np.cumsum([x.size for x in xs], dtype=np.uint64)
    return np.concatenate(xs), offsets, np.array(srs, np.uint32), note, units


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    subprocess.run(["make", "-s", "-C", str(ROOT / "oracle"), "-j8"], check=True)
    jobs = host_jobs()
    x, offs, srs, note, units = cpu_sample(args.workload, jobs)  # one track per worker and step: a bounded sample of the workload
    for _ in range(max(args.warmup, 0) and 1):  # one warm-up pass is enough for a CPU code (bounded run time)
        oracle_batch(x, offs, srs, jobs)
    times = [oracle_batch(x, offs, srs, jobs) for _ in range(args.steps)]
    ms = 1000.0 * sum(times) / len(times)
    val = units / (ms / 1000.0)
    metric, desc = WORKLOADS[args.workload]
    line = {
        "impl": "reference", "metric": metric, "value": val, "unit": "tracks/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": desc, "tracks_per_step": jobs,
                   "note": "CPU oracle port of stratum-dsp 1.0.0 (Rust toolchain absent), std::thread pool over tracks; its scalar FFT is about 4x slower "
                           "than rustfft's SIMD, so ratios against this arm flatter the GPU by about that factor (BASELINE.md)"},
        "cpu_baseline": {"value": val, "unit": "tracks/s", "cores": jobs, "kind": "port", "per_worker": val / jobs, "sample": f"{note} per step, {args.steps} steps"},
        "e2e": {"value": val, "unit": "tracks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


class Pinned:
    """Page-locked host array owned by this script (numpy storage registered with cudaHostRegister), released explicitly:
    torch's pinned-memory allocator caches freed blocks, which would keep hundreds of gigabytes locked between the legs."""

    def __init__(self, torch, n_elems: int, np_dtype):
        self.torch = torch
        item = np.dtype(np_dtype).itemsize
        raw = np.empty(n_elems + 4096 // item, dtype=np_dtype)  # page-aligned view (cudaHostRegister pins whole pages)
        skip = (-raw.ctypes.data % 4096) // item
        self.raw = raw
        self.arr = raw[skip:skip + n_elems]
        self.registered = False
        rc = torch.cuda.cudart().cudaHostRegister(self.arr.ctypes.data, self.arr.nbytes, 0)
        if int(rc) != 0:
            self.arr = None
            raise MemoryError(f"cudaHostRegister failed ({rc})")
        self.registered = True
        self.tensor = torch.from_numpy(self.arr)

    def free(self):
        if self.registered:
            self.torch.cuda.synchronize()
            self.torch.cuda.cudart().cudaHostUnregister(self.arr.ctypes.data)
            self.registered = False
        self.tensor = None
        self.arr = None
        self.raw = None


def pinned_empty(torch, n_elems: int, np_dtype):
    try:
        return Pinned(torch, n_elems, np_dtype)
    except (MemoryError, RuntimeError):
        return None


DUMP_CAP_BYTES = 60_000_000  # data bytes; with the .npy headers the dump stays below 64 MB
# per-track scalars of StratumResult; processing_time_ms is left out: it is a wall time and differs from run to run
DUMP_SCALARS = ("status", "bpm", "bpm_confidence", "key_is_minor", "key_index", "key_confidence", "key_clarity", "grid_stability",
                "duration_seconds", "sample_rate", "onset_method_consensus", "warnings", "flags", "tempogram_multi_res_triggered",
                "tempogram_multi_res_used", "tempogram_percussive_triggered", "tempogram_percussive_used", "trim_start", "trim_end",
                "time_sig_beats_per_bar", "beats_refined", "n_tempogram_candidates")
# per-track arrays: (pointer field, count field, dtype written)
DUMP_ARRAYS = (("beats", "n_beats", np.float32), ("downbeats", "n_downbeats", np.float32), ("bars", "n_bars", np.float32),
               ("onsets", "n_onsets", np.float64), ("hmm_beat_frames", "n_hmm_beat_frames", np.float64))


def dump_outputs(results, out_dir, seed: int = 0) -> int:
    """Writes the StratumResult array of one batch call as out_dir/<name>.npy, for comparing two builds output for output.

    Scalars are one float64 per track (integers stay exact).  A per-track array is written concatenated in track order with
    <name>_offsets.npy (track i = <name>[offsets[i]:offsets[i+1]]); tempogram_candidates has one row of (bpm, score, fft_norm,
    autocorr_norm, selected) per candidate.  An array that no track returned is not written: tempogram candidates, for one, exist only
    when the configuration emits them (n_tempogram_candidates is -1 otherwise).  If the whole batch exceeds DUMP_CAP_BYTES, a fixed,
    seeded sample of tracks is written; track_index.npy names the tracks written.  Returns the number of bytes written."""
    def arr(r, ptr, n, dtype):
        return np.ctypeslib.as_array(getattr(r, ptr), shape=(n,)).astype(dtype) if n and getattr(r, ptr) else np.zeros(0, dtype)

    def cands(r):
        n = max(r.n_tempogram_candidates, 0)
        return np.array([[c.bpm, c.score, c.fft_norm, c.autocorr_norm, c.selected] for c in r.tempogram_candidates[:n]], np.float32).reshape(n, 5)

    n = len(results)
    per_track = np.array([8 * (len(DUMP_SCALARS) + 1 + 6) + 4 * (r.n_beats + r.n_downbeats + r.n_bars) + 8 * (r.n_onsets + r.n_hmm_beat_frames)
                          + 20 * max(r.n_tempogram_candidates, 0) for r in results], np.int64)
    idx = np.arange(n)
    if per_track.sum() > DUMP_CAP_BYTES:
        order = np.random.default_rng(seed).permutation(n)
        idx = np.sort(order[np.cumsum(per_track[order]) <= DUMP_CAP_BYTES])
    picked = [results[int(i)] for i in idx]
    out = {"track_index": idx.astype(np.float64)}
    for f in DUMP_SCALARS:
        out[f] = np.array([getattr(r, f) for r in picked], np.float64)
    parts = {f: [arr(r, f, getattr(r, cnt), dt) for r in picked] for f, cnt, dt in DUMP_ARRAYS}
    parts["tempogram_candidates"] = [cands(r) for r in picked]
    for f, p in parts.items():
        if sum(len(a) for a in p) == 0:
            continue
        out[f"{f}_offsets"] = np.concatenate([[0], np.cumsum([len(a) for a in p])]).astype(np.float64)
        out[f] = np.concatenate(p)
    Path(out_dir).mkdir(parents=True, exist_ok=True)
    for name, a in out.items():
        np.save(Path(out_dir) / f"{name}.npy", a)
    return sum(a.nbytes for a in out.values())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--tracks", type=int, default=0, help="tracks per GPU and step (default: 1024 for c2 = BASELINE.json configs[1], 256 for c5, 1 for c4)")
    ap.add_argument("--e2e-tracks", type=int, default=0, help="tracks per GPU of the host-buffer (e2e) legs (default: the whole batch)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-multi-device-call", action="store_true", help="skip the one-process, one-call multi-device e2e leg at N > 1")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step (rank 0's tracks) as DIR/<name>.npy; the inputs are the same on every run")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the CUDA path's results; the reference arm has none to write")
    if args.impl == "reference":
        run_reference(args)
        return

    import torch
    import stratum_dsp_b200 as S

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not S.LIB_PATH.exists():
        raise SystemExit("libstratum_b200.so is missing — run __graft_entry__.build(); there is no fallback path")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    numa_note = bind_to_gpu_numa(local_rank)
    dist = None
    host_group = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(minutes=40))
        # host-side group: ranks that wait for rank 0's multi-device call must not spin in an NCCL kernel on the GPUs it measures
        host_group = dist.new_group(backend="gloo", timeout=datetime.timedelta(minutes=40))

    def barrier():
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        torch.cuda.synchronize()

    wl = args.workload
    metric, wl_desc = WORKLOADS[wl]
    nt = args.tracks or {"c2": 1024, "c5": 256, "c4": 1}[wl]
    lens, srs, rows, want_bpm = workload_layout(wl, rank * nt, nt)
    offsets = np.zeros(nt + 1, np.uint64)
    offsets[1:] = np.cumsum(lens, dtype=np.uint64)
    total_samples = int(offsets[-1])
    # ---- device-resident batch: generated on the device, outside the timed region ----
    buf = torch.empty(total_samples, dtype=torch.float32, device="cuda")
    fill_device(S, torch, wl, buf, offsets, lens, srs, rows, local_rank)

    waves = [1]

    def step():
        res = S.analyze_batch_device(buf.data_ptr(), offsets, srs, None, local_rank, convert=False)
        ms = S.last_call_device_ms()
        waves[0] = max(1, S.last_call_waves())
        return res, ms

    for _ in range(args.warmup):
        res, _ms = step()
        S.free_results(res)
    S.stage_timing(True)
    S.stage_times(reset=True)
    sampler = ClockSampler(local_rank)
    barrier()
    sampler.start()
    launches0 = S.launch_count()
    t0 = time.perf_counter()
    dev_ms = 0.0
    last = None
    for _ in range(args.steps):
        if last is not None:
            S.free_results(last)
        last, ms = step()
        dev_ms += ms
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1000.0
    launches = S.launch_count() - launches0
    clocks = sampler.stop()
    stages = S.stage_times(reset=True)
    S.stage_timing(False)
    # sanity on the last step's results (no oracle here: parity lives in tests/ and smoke())
    ok = sum(1 for r in last if r.status == 0)
    bpm_hit = 0
    for i, r in enumerate(last):
        b, t = r.bpm, float(want_bpm[i])
        tol = 2.0 if wl != "c4" else 6.0  # the mix drifts 120 -> 128
        if r.status == 0 and b > 0 and min(abs(b - t), abs(2 * b - t), abs(b - 2 * t)) <= tol:
            bpm_hit += 1
    n_escalated = sum(1 for r in last if r.status == 0 and r.tempogram_multi_res_triggered == 1)
    if args.dump_outputs and rank == 0:
        dump_outputs(last, args.dump_outputs)
    S.free_results(last)
    L = S.lib()
    L.stratum_b200_fp32_peak_tflops.restype = C.c_double
    fp32_peak = float(L.stratum_b200_fp32_peak_tflops(C.c_int32(local_rank)))

    # ---- e2e, per rank: host buffers through the reference-facing call on this rank's GPU ----
    e2e = None
    ne = min(args.e2e_tracks or nt, nt)
    if not args.no_e2e:
        host = None
        while host is None:  # a box with little lockable host memory gets a smaller (still pinned) e2e batch rather than no number — and says so
            host = pinned_empty(torch, int(offsets[ne]), np.float32)
            if host is None:
                if ne <= 1:
                    raise SystemExit("cannot pin host memory for the e2e leg")
                ne = max(1, ne // 2)
        host.tensor.copy_(buf[: int(offsets[ne])])
        torch.cuda.synchronize()
        hnp = host.arr
        eoff = np.ascontiguousarray(offsets[: ne + 1])
        srs_e = np.ascontiguousarray(srs[:ne])
        dev1 = (C.c_int32 * 1)(local_rank)

        def host_step():
            # the reference-facing C-ABI call itself (include/stratum_b200.h): host samples in, StratumResult array out
            res = (S.StratumResult * ne)()
            st = S.lib().stratum_b200_analyze_batch(hnp.ctypes.data, eoff.ctypes.data_as(C.POINTER(C.c_uint64)), srs_e.ctypes.data_as(C.POINTER(C.c_uint32)), ne,
                                                    None, dev1, 1, res)
            assert st == 0, S.last_error()
            n_ok = sum(1 for r in res if r.status == 0)
            S.free_results(res)
            return n_ok

        # pinned H2D rate of this box (outside the timed region): the ceiling of the f32 leg is this rate / bytes per track
        pn = min(int(offsets[ne]), 32 * N_SAMPLES)
        probe = torch.empty(pn, dtype=torch.float32, device="cuda")
        probe.copy_(host.tensor[:pn], non_blocking=True)
        torch.cuda.synchronize()
        tb0 = time.perf_counter()
        probe.copy_(host.tensor[:pn], non_blocking=True)
        torch.cuda.synchronize()
        h2d_gbs = pn * 4 / (time.perf_counter() - tb0) / 1e9
        del probe
        host_step()  # warm-up (staging buffer allocation)
        h0, d0 = S.transfer_bytes()
        barrier()
        te0 = time.perf_counter()
        e_steps = args.steps
        for _ in range(e_steps):
            host_step()
        barrier()
        e_ms = (time.perf_counter() - te0) * 1000.0 / e_steps
        h1, d1 = S.transfer_bytes()
        e2e = {"tracks_per_step": ne, "ms_per_step": e_ms, "h2d": (h1 - h0) // e_steps, "d2h": (d1 - d0) // e_steps, "h2d_gbs": h2d_gbs}
        # the decoder-side entry (16-bit PCM uploaded as is, converted on the device): half the H2D bytes
        hnp = None
        host.free()  # the f32 buffer is unpinned before the PCM one is pinned
        pcm = pinned_empty(torch, int(offsets[ne]), np.int16)
        if pcm is not None:
            sl = 8 * N_SAMPLES
            for a in range(0, int(offsets[ne]), sl):  # converted in slices: the analysis arenas own most of the device memory
                b = min(a + sl, int(offsets[ne]))
                pcm.tensor[a:b].copy_((buf[a:b] * 32767.0).round().clamp_(-32768, 32767).to(torch.int16))
            torch.cuda.synchronize()
            pnp = pcm.arr
            chans = np.ones(ne, np.uint32)

            def pcm_step():
                res = (S.StratumResult * ne)()
                st = S.lib().stratum_b200_analyze_batch_pcm16(pnp.ctypes.data, eoff.ctypes.data_as(C.POINTER(C.c_uint64)), srs_e.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                              chans.ctypes.data_as(C.POINTER(C.c_uint32)), ne, None, dev1, 1, res)
                assert st == 0, S.last_error()
                S.free_results(res)

            pcm_step()
            barrier()
            tp0 = time.perf_counter()
            for _ in range(e_steps):
                pcm_step()
            barrier()
            e2e["pcm16_ms_per_step"] = (time.perf_counter() - tp0) * 1000.0 / e_steps
            pnp = None
            pcm.free()
        else:
            barrier()
            barrier()
            e2e["pcm16_ms_per_step"] = 0.0

    # ---- CPU baseline: the oracle port on this box's host cores, bounded sample (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            subprocess.run(["make", "-s", "-C", str(ROOT / "oracle"), "-j8"], check=True)
            jobs = host_jobs()
            x, offs_c, srs_c, note, units = cpu_sample(wl, jobs)
            sec = oracle_batch(x, offs_c, srs_c, jobs)
            # the north-star target is stated against ONE reference worker: time it on its own (3 tracks, 1 thread)
            n1 = min(3, jobs)
            sec1 = oracle_batch(x[: int(offs_c[n1])], offs_c[: n1 + 1], srs_c[:n1], 1)
            units1 = units * n1 / jobs
            cpu = {"value": units / sec, "unit": "tracks/s", "cores": jobs, "kind": "port", "per_worker": units / sec / jobs,
                   "single_worker": {"value": units1 / sec1, "unit": "tracks/s", "cores": 1, "sample": f"the first {n1} tracks of the sample on one thread, {sec1:.1f} s wall"},
                   "sample": f"{note}, one per thread, {sec:.1f} s wall (CPU oracle, -O3)",
                   "note": "oracle port, scalar FFT: about 4x slower per worker than the Rust crate's rustfft SIMD path (BASELINE.md), so GPU/CPU ratios against it flatter the GPU by about that factor"}
        except Exception as e:  # the baseline is a reported number, never a reason to lose the GPU measurement
            cpu = {"value": None, "unit": "tracks/s", "cores": 0, "kind": "port", "sample": f"failed: {e}"}

    # ---- reduce over ranks: max time, summed units ----
    ms_step = dev_ms / args.steps
    wall_step = wall_ms / args.steps
    e_ms_step = e2e["ms_per_step"] if e2e else 0.0
    p_ms_step = e2e["pcm16_ms_per_step"] if e2e else 0.0
    ne_min = ne
    if dist:
        t = torch.tensor([ms_step, wall_step, e_ms_step, p_ms_step], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step, wall_step, e_ms_step, p_ms_step = (float(v) for v in t.tolist())
        c = torch.tensor([ok, bpm_hit, launches, n_escalated, total_samples], dtype=torch.int64, device="cuda")
        dist.all_reduce(c, op=dist.ReduceOp.SUM)
        ok, bpm_hit, launches, n_escalated, total_samples_all = (int(v) for v in c.tolist())
        m = torch.tensor([ne], dtype=torch.int64, device="cuda")
        dist.all_reduce(m, op=dist.ReduceOp.MIN)
        ne_min = int(m.item())
    else:
        total_samples_all = total_samples

    # ---- e2e, one call over all devices (rank 0; the other ranks release their GPUs and wait) ----
    multi = None
    if world > 1 and e2e is not None and not args.no_multi_device_call and wl != "c4":
        del buf
        S.shutdown()
        torch.cuda.empty_cache()
        barrier()
        if rank == 0:
            try:
                multi = multi_device_call(S, torch, wl, world, ne_min, args)
            except Exception as e:  # reported, never fatal for the rest of the line
                multi = {"error": f"{type(e).__name__}: {e}"}
            S.shutdown()
        torch.cuda.synchronize()
        dist.barrier(group=host_group)  # waits on the host: the other GPUs stay idle while rank 0 drives them

    if rank == 0:
        peak, peak_src = load_peaks()
        total_tracks = nt * world
        value = total_tracks / (ms_step / 1000.0)
        algo_bytes_step = 4 * total_samples  # SURVEY.md §8(d): one read of the input samples (this rank's share)
        # dominant kernel of the step, by device time on the launching stream.  Only single-kernel stages qualify: the
        # tail stages of the tempo path (tempograms, final BPM, beats, legacy, energy onsets) run on the second stream beside
        # the key path, so their event spans include time spent waiting for SM slots and say nothing about kernel cost.
        single = {k: v for k, v in stages.items() if k in ("stft_8192_key", "key_mask", "stft_2048_hop512")}
        dom = max(single, key=single.get) if single else (max(stages, key=stages.get) if stages else None)
        roof = None
        if dom:
            k_ms = stages[dom] / args.steps  # per step (all waves of the step)
            launches_per_step = waves[0]     # one launch of the kernel per wave
            ach = algo_bytes_step / (k_ms / 1000.0) / 1e9  # = per-launch bytes / per-launch time
            traffic, traffic_all = None, None
            tp = ROOT / "profiles" / "roofline_traffic.json"
            if tp.exists():  # DRAM bytes per 3-minute track from the committed `ncu --set full` captures -> bytes per launch
                try:
                    tj = json.loads(tp.read_text())
                    scale = total_samples / N_SAMPLES / launches_per_step  # 3-minute-track equivalents per launch
                    per_track = tj.get(dom, {}).get("dram_bytes_per_track")
                    traffic = per_track * scale if per_track else None
                    traffic_all = {k: v["dram_bytes_per_track"] * scale for k, v in tj.items() if isinstance(v, dict) and v.get("dram_bytes_per_track")}
                except Exception:
                    traffic = None
            frames_key = sum(max(0, (int(n) - 8192) // 512 + 1) for n in lens)
            frames_base = sum(max(0, (int(n) - 2048) // 512 + 1) for n in lens)
            roof = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                    "traffic_by_kernel": traffic_all,
                    "peak_source": peak_src, "algorithmic_bytes_per_step": algo_bytes_step, "kernel_ms_per_step": k_ms,
                    "launches_per_step": launches_per_step, "algorithmic_bytes_per_launch": algo_bytes_step / launches_per_step,
                    "kernel_ms_per_launch": k_ms / launches_per_step,
                    "share_of_step": k_ms / ms_step,
                    "note": "path is FP32/shared-memory bound (SURVEY §8d: ~315 flop/B); the HBM fraction is reported as the contract asks",
                    "fp32_tflops_key_stft": (frames_key * FLOPS_KEY_FRAME / (stages["stft_8192_key"] / args.steps / 1000.0) / 1e12) if "stft_8192_key" in stages else None}
            # second denominator (SURVEY §8d): STFT flops of the whole step by the 5 N log2 N convention against the measured FMA rate
            esc_frac = n_escalated / max(1, ok)
            step_flops = frames_base * FLOPS_BASE_FRAME * (1.0 + 2.5 * esc_frac) + frames_key * FLOPS_KEY_FRAME
            ach_tf = step_flops / (ms_step / 1000.0) / 1e12
            roof["fp32"] = {"achieved": ach_tf, "peak": fp32_peak or None, "unit": "TFLOP/s", "frac": (ach_tf / fp32_peak) if fp32_peak else None,
                            "peak_source": "measured: FMA microbenchmark of this run (stratum_b200_fp32_peak_tflops), 2 flops per FMA",
                            "flops_per_step": step_flops, "escalated_tracks": n_escalated,
                            "note": "STFT flops only (5 N log2 N for the complex transform of N points; the kernels use the real-input packing, "
                                    "so they execute about half of that; an escalated track adds hop-256 and hop-1024 passes = 2.5x its hop-512 frames); "
                                    "the path compiles with -fmad=false, FMAs only inside the FFT"}
        e2e_out = None
        if e2e:
            per_rank = {"value": ne_min * world / (e_ms_step / 1000.0), "unit": "tracks/s", "tracks_per_gpu": ne_min, "ms_per_step": e_ms_step,
                        "pcm16_value": (ne_min * world / (p_ms_step / 1000.0)) if p_ms_step > 0 else None,
                        "note": "N processes, each calling stratum_b200_analyze_batch on its own GPU with its own pinned host batch; max time over ranks"}
            if world == 1:
                head = dict(per_rank)
                head["note"] = "one process, one call of stratum_b200_analyze_batch on pinned host f32 samples: H2D of the samples and D2H of the results inside the timed region"
            elif multi and "value" in multi:
                head = multi
            else:
                head = dict(per_rank)
                head["note"] = "per-rank calls (the one-call multi-device leg did not run: " + (multi or {}).get("error", "disabled") + ")"
            e2e_out = {"value": head["value"], "unit": "tracks/s", "h2d_bytes_per_step": int(head.get("h2d_bytes_per_step", e2e["h2d"] * world)),
                       "d2h_bytes_per_step": int(head.get("d2h_bytes_per_step", e2e["d2h"] * world)), "tracks_per_gpu": head.get("tracks_per_gpu", ne_min),
                       "ms_per_step": head["ms_per_step"], "pcm16_value": head.get("pcm16_value"), "pinned_h2d_gbs_rank0": e2e["h2d_gbs"],
                       "call": "stratum_b200_analyze_batch(device_ids=[0..N-1]) from one process" if world > 1 and multi and "value" in multi else "stratum_b200_analyze_batch, one process per GPU",
                       "note": head["note"], "per_rank": per_rank}
            e2e_out["h2d_gbs_aggregate"] = e2e_out["h2d_bytes_per_step"] / (e2e_out["ms_per_step"] / 1000.0) / 1e9
            e2e_out["h2d_note"] = ("pinned_h2d_gbs_rank0 is a plain pinned torch copy timed while every rank does the same: times N it is the host's aggregate "
                                   "host-to-device rate, the ceiling of the f32 leg (31.75 MB per track); pcm16_value moves half the bytes")
            if multi and "value" in multi:
                e2e_out["multi_device_call"] = {k: v for k, v in multi.items() if k not in ("note",)}
        line = {
            "metric": metric, "value": value, "unit": "tracks/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl_desc, "tracks_per_gpu_per_step": nt, "samples_per_gpu_per_step": total_samples,
                       "audio_hours_per_gpu_per_step": float(sum(float(n) / float(s) for n, s in zip(lens, srs)) / 3600.0),
                       "l2": f"inputs ({4 * total_samples / 1e9:.1f} GB per GPU) far larger than L2; no flush needed",
                       "timing": "CUDA events on the library stream around each batch call, max over ranks", "host_placement": numa_note},
            "ms_per_track": ms_step / nt, "wall_ms_per_step": wall_step,
            "gpu_launches": launches, "clocks": clocks,
            "stages_ms_per_step": {k: v / args.steps for k, v in stages.items()},
            "stages_note": "CUDA-event spans per stream; onsets_energy, legacy_bpm, multires_tempogram, final_bpm and beats run on the second stream "
                           "beside other kernels (late split), so their spans overlap the key-path stages and do not add up to the step; "
                           "host_escalation = host time spent waiting for the escalated-track count while the device is busy (not idle device time)",
            "results_ok": ok, "bpm_within_2_or_octave": bpm_hit, "tracks_total": total_tracks, "escalated_tracks": n_escalated,
            "roofline": roof,
            "cpu_baseline": cpu,
            "e2e": e2e_out,
        }
        print(json.dumps(line), flush=True)
    if dist:
        dist.barrier()
        dist.destroy_process_group()


def multi_device_call(S, torch, wl, world, ne, args):
    """Rank 0, every GPU of the box free: one process, one stratum_b200_analyze_batch call over device_ids = [0 .. world-1] on
    world x ne pinned host tracks (the same per-GPU batch as at N = 1; halved, and reported, only if the host cannot pin it)."""
    per_gpu = ne
    host = None
    while host is None:
        lens, srs, rows, _ = workload_layout(wl, 0, per_gpu * world)
        offsets = np.zeros(per_gpu * world + 1, np.uint64)
        offsets[1:] = np.cumsum(lens, dtype=np.uint64)
        host = pinned_empty(torch, int(offsets[-1]), np.float32)
        if host is None:
            if per_gpu <= 16:
                raise RuntimeError("cannot pin the host batch")
            per_gpu //= 2
    n_all = per_gpu * world
    # fill through GPU 0 in slices of 64 tracks (generator on the device, D2H into the pinned batch); outside the timed region
    for a in range(0, n_all, 64):
        b = min(a + 64, n_all)
        tmp = torch.empty(int(offsets[b] - offsets[a]), dtype=torch.float32, device="cuda")
        rel = offsets[a:b + 1] - offsets[a]
        fill_device(S, torch, wl, tmp, rel, lens[a:b], srs[a:b], rows[a:b] if rows is not None else None, 0)
        host.tensor[int(offsets[a]):int(offsets[b])].copy_(tmp)
        del tmp
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    hnp = host.arr
    devs = (C.c_int32 * world)(*range(world))
    srs_c = np.ascontiguousarray(srs)

    def call():
        res = (S.StratumResult * n_all)()
        st = S.lib().stratum_b200_analyze_batch(hnp.ctypes.data, offsets.ctypes.data_as(C.POINTER(C.c_uint64)), srs_c.ctypes.data_as(C.POINTER(C.c_uint32)), n_all,
                                                None, devs, world, res)
        assert st == 0, S.last_error()
        n_ok = sum(1 for r in res if r.status == 0)
        S.free_results(res)
        return n_ok

    call()  # warm-up: contexts, arenas and staging buffers of every device
    steps = args.steps
    h0, d0 = S.transfer_bytes()
    t0 = time.perf_counter()
    n_ok = 0
    for _ in range(steps):
        n_ok = call()
    ms = (time.perf_counter() - t0) * 1000.0 / steps
    h1, d1 = S.transfer_bytes()
    out = {"value": n_all / (ms / 1000.0), "unit": "tracks/s", "tracks_per_gpu": per_gpu, "tracks_per_call": n_all, "ms_per_step": ms, "results_ok": n_ok,
           "h2d_bytes_per_step": (h1 - h0) // steps, "d2h_bytes_per_step": (d1 - d0) // steps,
           "note": f"one process, one call of stratum_b200_analyze_batch(device_ids=[0..{world - 1}]) on {n_all} pinned host f32 tracks ({per_gpu} per GPU): "
                   "the library shards by track, one host thread + one uploader thread per device; H2D of the samples and D2H of the results inside the timed region"}
    # PCM16 through the same path: convert through GPU 0 slice by slice into a pinned int16 batch
    hnp = None
    pcm = pinned_empty(torch, int(offsets[-1]), np.int16)
    if pcm is None:
        host.free()
    else:
        sl = 16 * N_SAMPLES
        for a in range(0, int(offsets[-1]), sl):
            b = min(a + sl, int(offsets[-1]))
            d = host.tensor[a:b].cuda(non_blocking=True)
            pcm.tensor[a:b].copy_((d * 32767.0).round().clamp_(-32768, 32767).to(torch.int16))
            del d
        torch.cuda.synchronize()
        host.free()
        torch.cuda.empty_cache()
        pnp = pcm.arr
        chans = np.ones(n_all, np.uint32)

        def pcall():
            res = (S.StratumResult * n_all)()
            st = S.lib().stratum_b200_analyze_batch_pcm16(pnp.ctypes.data, offsets.ctypes.data_as(C.POINTER(C.c_uint64)), srs_c.ctypes.data_as(C.POINTER(C.c_uint32)),
                                                          chans.ctypes.data_as(C.POINTER(C.c_uint32)), n_all, None, devs, world, res)
            assert st == 0, S.last_error()
            S.free_results(res)

        pcall()
        t0 = time.perf_counter()
        for _ in range(steps):
            pcall()
        pms = (time.perf_counter() - t0) * 1000.0 / steps
        out["pcm16_value"] = n_all / (pms / 1000.0)
        out["pcm16_ms_per_step"] = pms
        pnp = None
        pcm.free()
    return out


if __name__ == "__main__":
    main()
