"""bench.py --dump-outputs: the results of the last timed step as .npy files, laid out so that two builds can be compared
output for output."""
import ctypes as C
import json
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import bench
import stratum_dsp_b200 as S

ROOT = Path(__file__).resolve().parent.parent


def _fake_results(n_beats_per_track):
    res = (S.StratumResult * len(n_beats_per_track))()
    keep = []
    for i, nb in enumerate(n_beats_per_track):
        r = res[i]
        r.status, r.bpm, r.key_index, r.trim_end, r.processing_time_ms = 0, 100.0 + i, i % 12, 7_938_000 - i, 12.5
        beats = (C.c_float * nb)(*[0.5 * k + i for k in range(nb)])
        onsets = (C.c_int64 * 3)(i, 1000 + i, 2**40 + i)
        cand = (S.StratumTempoCandidate * 2)(S.StratumTempoCandidate(120.0 + i, 0.9, 1.0, 0.5, 1), S.StratumTempoCandidate(60.0, 0.1, 0.2, 0.3, 0))
        keep += [beats, onsets, cand]
        r.beats, r.n_beats = C.cast(beats, C.POINTER(C.c_float)), nb
        r.onsets, r.n_onsets = C.cast(onsets, C.POINTER(C.c_int64)), 3
        r.tempogram_candidates, r.n_tempogram_candidates = C.cast(cand, C.POINTER(S.StratumTempoCandidate)), 2
    res[len(n_beats_per_track) - 1].status = 3  # a failed track: no arrays, no candidates
    res[len(n_beats_per_track) - 1].n_tempogram_candidates = -1
    return res, keep


def _load(d):
    return {p.stem: np.load(p) for p in Path(d).glob("*.npy")}


def test_dump_layout(tmp_path):
    res, _keep = _fake_results([4, 0, 7])
    res[2].beats, res[2].n_beats = None, 0
    res[2].onsets, res[2].n_onsets = None, 0
    res[2].tempogram_candidates = None
    bench.dump_outputs(res, tmp_path)
    d = _load(tmp_path)
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert "processing_time_ms" not in d and set(bench.DUMP_SCALARS) <= set(d)
    assert list(d["track_index"]) == [0, 1, 2] and list(d["status"]) == [0, 0, 3] and list(d["bpm"]) == [100, 101, 102]
    assert list(d["trim_end"]) == [7_938_000, 7_937_999, 7_937_998]
    assert d["beats"].dtype == np.float32 and list(d["beats_offsets"]) == [0, 4, 4, 4]
    assert list(d["beats"]) == [0.0, 0.5, 1.0, 1.5]
    assert d["onsets"].dtype == np.float64 and list(d["onsets"]) == [0, 1000, 2**40, 1, 1001, 2**40 + 1]  # int64 exact in float64
    assert d["tempogram_candidates"].shape == (4, 5) and list(d["tempogram_candidates_offsets"]) == [0, 2, 4, 4]
    assert list(d["n_tempogram_candidates"]) == [2, 2, -1]
    assert all(a.size > 0 for a in d.values())  # bars and downbeats: no track returned any, so no empty file
    assert not {"bars", "bars_offsets", "downbeats", "downbeats_offsets"} & set(d)


def test_dump_without_tempogram_candidates_writes_no_empty_file(tmp_path):
    # the default configuration does not emit candidates: every track reports -1 and there is nothing to write
    res, _keep = _fake_results([3, 5])
    for r in res:
        r.tempogram_candidates, r.n_tempogram_candidates = None, -1
    bench.dump_outputs(res, tmp_path)
    d = _load(tmp_path)
    assert "tempogram_candidates" not in d and "tempogram_candidates_offsets" not in d
    assert list(d["n_tempogram_candidates"]) == [-1, -1] and all(a.size > 0 for a in d.values())


def test_dump_over_the_cap_writes_a_fixed_sample(tmp_path, monkeypatch):
    res, _keep = _fake_results([1000] * 40)
    monkeypatch.setattr(bench, "DUMP_CAP_BYTES", 10 * 5000)
    assert bench.dump_outputs(res, tmp_path / "a") <= 10 * 5000
    bench.dump_outputs(res, tmp_path / "b")
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    idx = a["track_index"].astype(int)
    assert 0 < len(idx) < 40 and list(idx) == sorted(idx) and np.array_equal(a["bpm"], 100.0 + idx)
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)


def test_dump_with_the_reference_arm_is_rejected(tmp_path):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path / "d")],
                         capture_output=True, text=True)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_bench_dump_is_what_the_timed_path_returns(tmp_path):
    out = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--tracks", "3", "--steps", "2", "--warmup", "1", "--no-e2e", "--no-cpu-baseline",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, cwd=tmp_path)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["tracks_total"] == 3
    d = _load(tmp_path)
    assert all(a.size > 0 for a in d.values()) and "tempogram_candidates" not in d  # the default configuration emits no candidates
    import torch

    lens, srs, rows, _ = bench.workload_layout("c2", 0, 3)
    offsets = np.zeros(4, np.uint64)
    offsets[1:] = np.cumsum(lens, dtype=np.uint64)
    buf = torch.empty(int(offsets[-1]), dtype=torch.float32, device="cuda")
    bench.fill_device(S, torch, "c2", buf, offsets, lens, srs, rows, 0)
    want = S.analyze_batch_device(buf.data_ptr(), offsets, srs, None, 0)
    assert list(d["track_index"]) == [0, 1, 2] and list(d["status"]) == [0, 0, 0]
    for i, r in enumerate(want):
        assert d["bpm"][i] == np.float32(r.bpm) and d["key_clarity"][i] == np.float32(r.key_clarity)
        assert (d["key_is_minor"][i], d["key_index"][i]) == (r.key.is_minor, r.key.index)
        b0, b1 = d["beats_offsets"][i:i + 2].astype(int)
        assert np.array_equal(d["beats"][b0:b1], r.beat_grid.beats)
        o0, o1 = d["onsets_offsets"][i:i + 2].astype(int)
        assert np.array_equal(d["onsets"][o0:o1], r.onsets.astype(np.float64))
