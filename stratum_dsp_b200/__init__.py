"""stratum_dsp_b200 — host-side mirror of stratum-dsp's analysis API over the B200 C ABI.

The product is ``_build/libstratum_b200.so`` (hand-written sm_100a kernels + C ABI, see
``include/stratum_b200.h``).  This module is the thin binding a caller uses from Python and mirrors
the reference's public surface (src/lib.rs:52-56):

    analyze_audio(samples, sample_rate, config)  -> AnalysisResult      (src/lib.rs:86-90)
    compute_confidence(result)                   -> AnalysisConfidence  (src/analysis/confidence.rs:121)
    analyze_batch(tracks, sample_rates, config)  -> [AnalysisResult]    (examples/analyze_batch.rs:260-326)
    AnalysisConfig / AnalysisError / Key         (src/config.rs, src/error.rs, src/analysis/result.rs)

There is no CPU fallback and no oracle on this path: if the shared library is missing or no CUDA
device is usable, every compute call raises.
"""
from __future__ import annotations

import ctypes as C
import subprocess
from dataclasses import dataclass, field
from pathlib import Path
from typing import Iterable, Sequence

import numpy as np

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "_build" / "libstratum_b200.so"

ABI_VERSION = 2

# StratumStatus / AnalysisError variants (src/error.rs:7-22)
OK, INVALID_INPUT, DECODING_ERROR, PROCESSING_ERROR, NOT_IMPLEMENTED, NUMERICAL_ERROR = range(6)
_ERR_NAMES = {1: "InvalidInput", 2: "DecodingError", 3: "ProcessingError", 4: "NotImplemented", 5: "NumericalError"}

WARN_BPM_FAILED, WARN_LOW_GRID_STABILITY, WARN_LOW_KEY_CONFIDENCE, WARN_LOW_KEY_CLARITY = 1, 2, 4, 8
FLAG_MULTIMODAL_BPM, FLAG_WEAK_TONALITY, FLAG_TEMPO_VARIATION, FLAG_ONSET_AMBIGUOUS = 1, 2, 4, 8
_FLAG_NAMES = {1: "MultimodalBpm", 2: "WeakTonality", 4: "TempoVariation", 8: "OnsetDetectionAmbiguous"}

NORM_PEAK, NORM_RMS, NORM_LOUDNESS = 0, 1, 2


class AnalysisError(Exception):
    """AnalysisError (src/error.rs:7-22): ``kind`` is the variant name, ``code`` the StratumStatus."""

    def __init__(self, code: int, message: str):
        self.code = code
        self.kind = _ERR_NAMES.get(code, "ProcessingError")
        self.message = message
        super().__init__(f"{self.kind}: {message}")


_f, _i, _u = C.c_float, C.c_int32, C.c_uint32


class StratumConfig(C.Structure):
    """Mirror of ``StratumConfig`` in include/stratum_b200.h (field order is the ABI)."""

    _fields_ = [
        ("abi_version", _u), ("min_amplitude_db", _f), ("normalization", _i), ("enable_normalization", _i),
        ("enable_silence_trimming", _i), ("enable_onset_consensus", _i), ("onset_threshold_percentile", _f),
        ("onset_consensus_tolerance_ms", _u), ("onset_consensus_weights", _f * 4), ("enable_hpss_onsets", _i),
        ("force_legacy_bpm", _i), ("enable_bpm_fusion", _i), ("enable_legacy_bpm_guardrails", _i),
        ("enable_tempogram_multi_resolution", _i), ("tempogram_multi_res_top_k", _u), ("tempogram_multi_res_w512", _f),
        ("tempogram_multi_res_w256", _f), ("tempogram_multi_res_w1024", _f), ("tempogram_multi_res_structural_discount", _f),
        ("tempogram_multi_res_double_time_512_factor", _f), ("tempogram_multi_res_margin_threshold", _f),
        ("tempogram_multi_res_use_human_prior", _i), ("enable_tempogram_percussive_fallback", _i),
        ("enable_tempogram_band_fusion", _i), ("tempogram_band_low_max_hz", _f), ("tempogram_band_mid_max_hz", _f),
        ("tempogram_band_high_max_hz", _f), ("tempogram_band_w_full", _f), ("tempogram_band_w_low", _f),
        ("tempogram_band_w_mid", _f), ("tempogram_band_w_high", _f), ("tempogram_band_seed_only", _i),
        ("tempogram_band_support_threshold", _f), ("tempogram_band_consensus_bonus", _f),
        ("tempogram_novelty_w_spectral", _f), ("tempogram_novelty_w_energy", _f), ("tempogram_novelty_w_hfc", _f),
        ("tempogram_novelty_local_mean_window", _u), ("tempogram_novelty_smooth_window", _u),
        ("enable_tempogram_mel_novelty", _i), ("tempogram_mel_n_mels", _u), ("tempogram_mel_fmin_hz", _f),
        ("tempogram_mel_fmax_hz", _f), ("tempogram_mel_max_filter_bins", _u), ("tempogram_mel_weight", _f),
        ("tempogram_superflux_max_filter_bins", _u), ("emit_tempogram_candidates", _i), ("tempogram_candidates_top_n", _u),
        ("legacy_bpm_preferred_min", _f), ("legacy_bpm_preferred_max", _f), ("legacy_bpm_soft_min", _f), ("legacy_bpm_soft_max", _f),
        ("legacy_bpm_conf_mul_preferred", _f), ("legacy_bpm_conf_mul_soft", _f), ("legacy_bpm_conf_mul_extreme", _f),
        ("min_bpm", _f), ("max_bpm", _f), ("bpm_resolution", _f), ("frame_size", _u), ("hop_size", _u), ("soft_mapping_sigma", _f),
        ("key_spectrogram_smooth_margin", _u), ("enable_key_frame_weighting", _i), ("key_min_tonalness", _f),
        ("key_tonalness_power", _f), ("key_energy_power", _f), ("enable_key_harmonic_mask", _i), ("key_harmonic_mask_power", _f),
        ("enable_key_stft_override", _i), ("key_stft_frame_size", _u), ("key_stft_hop_size", _u),
        ("enable_key_segment_voting", _i), ("key_segment_len_frames", _u), ("key_segment_hop_frames", _u),
        ("key_segment_min_clarity", _f), ("enable_key_hpcp", _i), ("key_hpcp_peaks_per_frame", _u), ("key_hpcp_num_harmonics", _u),
        ("key_hpcp_harmonic_decay", _f), ("key_hpcp_mag_power", _f),
        ("enable_key_hpss_harmonic", _i), ("enable_key_log_frequency", _i), ("enable_key_beat_synchronous", _i),
        ("enable_key_multi_scale", _i), ("enable_key_ensemble", _i), ("enable_key_median", _i),
        ("enable_key_tuning_compensation", _i), ("enable_key_edge_trim", _i), ("enable_key_mode_heuristic", _i),
        ("enable_key_hpcp_whitening", _i), ("enable_key_hpcp_bass_blend", _i), ("enable_key_minor_harmonic_bonus", _i),
        ("chroma_sharpening_power", _f), ("hpss_margin", _u), ("soft_chroma_mapping", _i),
        ("enable_key_spectrogram_time_smoothing", _i),
        ("key_template_set", _i), ("key_edge_trim_fraction", _f), ("key_mode_third_ratio_margin", _f),
        ("key_mode_flip_min_score_ratio", _f), ("key_minor_leading_tone_bonus_weight", _f), ("key_ensemble_kk_weight", _f),
        ("key_ensemble_temperley_weight", _f), ("key_multi_scale_n_lengths", _u), ("key_multi_scale_lengths", _u * 8),
        ("key_multi_scale_hop", _u), ("key_multi_scale_min_clarity", _f), ("key_multi_scale_n_weights", _u),
        ("key_multi_scale_weights", _f * 8), ("key_median_segment_length_frames", _u), ("key_median_segment_hop_frames", _u),
        ("key_median_min_segments", _u), ("key_tuning_max_abs_semitones", _f), ("key_tuning_frame_step", _u),
        ("key_tuning_peak_rel_threshold", _f), ("key_hpss_frame_step", _u), ("key_hpss_time_margin", _u), ("key_hpss_freq_margin", _u),
        ("key_hpss_mask_power", _f), ("key_hpcp_whitening_smooth_bins", _u), ("key_hpcp_bass_fmin_hz", _f),
        ("key_hpcp_bass_fmax_hz", _f), ("key_hpcp_bass_weight", _f),
    ]


class StratumTempoCandidate(C.Structure):
    _fields_ = [("bpm", _f), ("score", _f), ("fft_norm", _f), ("autocorr_norm", _f), ("selected", _i)]


class StratumResult(C.Structure):
    _fields_ = [
        ("status", _i), ("error", C.c_char * 128), ("bpm", _f), ("bpm_confidence", _f), ("key_is_minor", _i), ("key_index", _u),
        ("key_confidence", _f), ("key_clarity", _f), ("grid_stability", _f),
        ("beats", C.POINTER(_f)), ("downbeats", C.POINTER(_f)), ("bars", C.POINTER(_f)),
        ("n_beats", _u), ("n_downbeats", _u), ("n_bars", _u),
        ("duration_seconds", _f), ("sample_rate", _u), ("processing_time_ms", _f), ("onset_method_consensus", _f),
        ("warnings", _u), ("flags", _u),
        ("tempogram_multi_res_triggered", _i), ("tempogram_multi_res_used", _i),
        ("tempogram_percussive_triggered", _i), ("tempogram_percussive_used", _i),
        ("trim_start", C.c_uint64), ("trim_end", C.c_uint64), ("onsets", C.POINTER(C.c_int64)), ("n_onsets", _u),
        ("hmm_beat_frames", C.POINTER(_i)), ("n_hmm_beat_frames", _u), ("time_sig_beats_per_bar", _i), ("beats_refined", _i),
        ("tempogram_candidates", C.POINTER(StratumTempoCandidate)), ("n_tempogram_candidates", _i),
    ]


class StratumConfidence(C.Structure):
    _fields_ = [("bpm_confidence", _f), ("key_confidence", _f), ("grid_stability", _f), ("overall_confidence", _f), ("flags", _u)]


class StratumLoudness(C.Structure):
    _fields_ = [
        ("status", _i), ("error", C.c_char * 128), ("sample_rate", _u), ("channels", _u), ("frames", C.c_uint64),
        ("integrated_lufs", C.c_double), ("momentary_max_lufs", C.c_double), ("short_term_max_lufs", C.c_double),
        ("loudness_range_lu", C.c_double), ("sample_peak", C.c_double), ("true_peak", C.c_double),
        ("n_momentary", _u), ("n_short_term", _u),
    ]


_lib: C.CDLL | None = None


def build(force: bool = False) -> Path:
    """Compile the CUDA extension in-tree (nvcc, sm_100a).  Cross-compiles without a GPU."""
    if force:
        subprocess.run(["make", "-s", "-C", str(_PKG), "clean"], check=True)
    subprocess.run(["make", "-s", "-C", str(_PKG), "-j8"], check=True)
    return LIB_PATH


def lib() -> C.CDLL:
    """The C-ABI library.  Raises if it has not been built — there is no fallback implementation."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise RuntimeError(f"{LIB_PATH} is missing: run stratum_dsp_b200.build() (nvcc) first; this package has no CPU fallback")
    L = C.CDLL(str(LIB_PATH))
    cfgp, resp = C.POINTER(StratumConfig), C.POINTER(StratumResult)
    u64p, u32p, i32p, f32p = C.POINTER(C.c_uint64), C.POINTER(_u), C.POINTER(_i), C.POINTER(_f)
    L.stratum_b200_config_default.argtypes = [cfgp]
    L.stratum_b200_config_default.restype = None
    L.stratum_b200_analyze_batch.argtypes = [C.c_void_p, u64p, u32p, _u, cfgp, i32p, _u, resp]
    L.stratum_b200_analyze_batch.restype = _i
    L.stratum_b200_analyze_batch_pcm16.argtypes = [C.c_void_p, u64p, u32p, u32p, _u, cfgp, i32p, _u, resp]
    L.stratum_b200_analyze_batch_pcm16.restype = _i
    L.stratum_b200_analyze_batch_device.argtypes = [C.c_void_p, u64p, u32p, _u, cfgp, _i, resp]
    L.stratum_b200_analyze_batch_device.restype = _i
    L.stratum_b200_analyze_audio.argtypes = [C.c_void_p, C.c_uint64, _u, cfgp, resp]
    L.stratum_b200_analyze_audio.restype = _i
    L.stratum_b200_compute_confidence.argtypes = [resp, C.POINTER(StratumConfidence)]
    L.stratum_b200_compute_confidence.restype = None
    L.stratum_b200_warning_strings.argtypes = [resp, C.c_char_p, C.c_size_t]
    L.stratum_b200_warning_strings.restype = _i
    L.stratum_b200_key_name.argtypes = [_i, _u, _i, C.c_char_p, C.c_size_t]
    L.stratum_b200_key_name.restype = _i
    L.stratum_b200_result_free.argtypes = [resp, _u]
    L.stratum_b200_result_free.restype = None
    L.stratum_b200_last_error.argtypes = [C.c_char_p, C.c_size_t]
    L.stratum_b200_last_error.restype = _i
    L.stratum_b200_launch_count.argtypes = []
    L.stratum_b200_launch_count.restype = C.c_uint64
    L.stratum_b200_device_count.argtypes = []
    L.stratum_b200_device_count.restype = _i
    L.stratum_b200_shutdown.argtypes = []
    L.stratum_b200_shutdown.restype = None
    L.stratum_b200_sizeof.argtypes = [_i]
    L.stratum_b200_sizeof.restype = C.c_size_t
    L.stratum_b200_stft.argtypes = [C.c_void_p, C.c_uint64, _u, _u, _f, C.c_void_p, C.c_uint64]
    L.stratum_b200_stft.restype = C.c_int64
    L.stratum_b200_synth_batch.argtypes = [C.c_void_p, _u, C.c_uint64, _u, f32p, _i]
    L.stratum_b200_synth_batch.restype = _i
    L.stratum_b200_debug_array.argtypes = [C.c_char_p, C.c_void_p, C.c_int64]
    L.stratum_b200_debug_array.restype = C.c_int64
    L.stratum_b200_debug_enable.argtypes = [_i]
    L.stratum_b200_debug_enable.restype = None
    L.stratum_b200_stage_times.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_double), _i]
    L.stratum_b200_stage_times.restype = _i
    L.stratum_b200_stage_times_reset.argtypes = []
    L.stratum_b200_stage_times_reset.restype = None
    L.stratum_b200_stage_timing_enable.argtypes = [_i]
    L.stratum_b200_stage_timing_enable.restype = None
    L.stratum_b200_last_call_device_ms.argtypes = []
    L.stratum_b200_last_call_device_ms.restype = C.c_double
    L.stratum_b200_last_call_waves.argtypes = []
    L.stratum_b200_last_call_waves.restype = _u
    L.stratum_b200_transfer_bytes.argtypes = [u64p, u64p]
    L.stratum_b200_transfer_bytes.restype = None
    loudp = C.POINTER(StratumLoudness)
    L.stratum_b200_loudness_batch_pcm.argtypes = [C.c_void_p, u64p, u32p, u32p, u32p, _u, i32p, _u, loudp]
    L.stratum_b200_loudness_batch_pcm.restype = _i
    L.stratum_b200_loudness_batch_pcm_device.argtypes = [C.c_void_p, u64p, u32p, u32p, u32p, _u, _i, loudp]
    L.stratum_b200_loudness_batch_pcm_device.restype = _i
    L.stratum_b200_loudness_albums_pcm.argtypes = [C.c_void_p, u64p, u32p, u32p, u32p, _u, u32p, _u, i32p, _u, loudp, loudp]
    L.stratum_b200_loudness_albums_pcm.restype = _i
    L.stratum_b200_loudness_albums_pcm_device.argtypes = [C.c_void_p, u64p, u32p, u32p, u32p, _u, u32p, _u, _i, loudp, loudp]
    L.stratum_b200_loudness_albums_pcm_device.restype = _i
    L.stratum_b200_analyze_loudness_pcm.argtypes = [C.c_void_p, u64p, u32p, u32p, u32p, _u, C.c_void_p, u32p, _u, i32p, _u, C.POINTER(StratumResult),
                                                    loudp, loudp]
    L.stratum_b200_analyze_loudness_pcm.restype = _i
    L.stratum_b200_debug_loudness_filters.argtypes = [_u, C.POINTER(C.c_double), f32p]
    L.stratum_b200_debug_loudness_filters.restype = _i
    if L.stratum_b200_sizeof(0) != C.sizeof(StratumConfig) or L.stratum_b200_sizeof(1) != C.sizeof(StratumResult) or \
            L.stratum_b200_sizeof(2) != C.sizeof(StratumConfidence) or L.stratum_b200_sizeof(3) != C.sizeof(StratumLoudness):
        raise RuntimeError("ctypes mirror of include/stratum_b200.h is out of date (struct size mismatch)")
    _lib = L
    return L


def last_error() -> str:
    buf = C.create_string_buffer(1024)
    lib().stratum_b200_last_error(buf, 1024)
    return buf.value.decode(errors="replace")


def _raise(code: int) -> None:
    raise AnalysisError(code, last_error())


class AnalysisConfig:
    """AnalysisConfig (src/config.rs:8-592) with the reference's field names; ``AnalysisConfig()`` is
    ``AnalysisConfig::default()`` (src/config.rs:594-744).  Unknown names raise AttributeError."""

    _names = {n for n, _ in StratumConfig._fields_}

    def __init__(self, **overrides):
        c = StratumConfig()
        lib().stratum_b200_config_default(C.byref(c))
        object.__setattr__(self, "_c", c)
        for k, v in overrides.items():
            setattr(self, k, v)

    # Vec<_> fields of the reference (config.rs:432-444) travel as a fixed array + count
    _vecs = {"key_multi_scale_lengths": "key_multi_scale_n_lengths", "key_multi_scale_weights": "key_multi_scale_n_weights"}

    def __getattr__(self, name):
        if name in AnalysisConfig._names:
            v = getattr(self._c, name)
            if name in AnalysisConfig._vecs:
                return list(v)[: getattr(self._c, AnalysisConfig._vecs[name])]
            return list(v) if name == "onset_consensus_weights" else v
        raise AttributeError(name)

    def __setattr__(self, name, value):
        if name not in AnalysisConfig._names:
            raise AttributeError(f"AnalysisConfig has no field {name!r}")
        if name == "onset_consensus_weights":
            for i, w in enumerate(value):
                self._c.onset_consensus_weights[i] = float(w)
        elif name in AnalysisConfig._vecs:
            value = list(value)
            if len(value) > 8:
                raise ValueError(f"{name}: at most 8 entries")
            arr = getattr(self._c, name)
            for i in range(8):
                arr[i] = (value[i] if i < len(value) else 0)
            setattr(self._c, AnalysisConfig._vecs[name], len(value))
        else:
            setattr(self._c, name, int(value) if isinstance(value, bool) else value)

    def clone(self) -> "AnalysisConfig":
        o = AnalysisConfig()
        C.memmove(C.byref(o._c), C.byref(self._c), C.sizeof(StratumConfig))
        return o


@dataclass(frozen=True)
class Key:
    """Key::Major(i) / Key::Minor(i) (src/analysis/result.rs:7-140)."""

    is_minor: bool
    index: int

    def name(self) -> str:
        buf = C.create_string_buffer(16)
        lib().stratum_b200_key_name(int(self.is_minor), self.index, 0, buf, 16)
        return buf.value.decode()

    def numerical(self) -> str:
        buf = C.create_string_buffer(16)
        lib().stratum_b200_key_name(int(self.is_minor), self.index, 1, buf, 16)
        return buf.value.decode()

    @property
    def id(self) -> int:
        return (12 if self.is_minor else 0) + self.index


@dataclass
class BeatGrid:
    beats: np.ndarray
    downbeats: np.ndarray
    bars: np.ndarray


@dataclass
class AnalysisMetadata:
    duration_seconds: float
    sample_rate: int
    processing_time_ms: float
    algorithm_version: str
    onset_method_consensus: float
    methods_used: list
    flags: list
    confidence_warnings: list
    tempogram_multi_res_triggered: bool | None
    tempogram_multi_res_used: bool | None
    tempogram_percussive_triggered: bool | None
    tempogram_percussive_used: bool | None
    tempogram_candidates: list | None = None  # [(bpm, score, fft_norm, autocorr_norm, selected)] when emit_tempogram_candidates


# AnalysisMetadata literals the reference writes at lib.rs:1603-1608 (the same three strings for every track)
ALGORITHM_VERSION = "0.1.0-alpha"
METHODS_USED = ("energy_flux", "chroma_extraction", "key_detection")


@dataclass
class AnalysisConfidence:
    bpm_confidence: float
    key_confidence: float
    grid_stability: float
    overall_confidence: float
    flags: list


@dataclass
class AnalysisResult:
    """AnalysisResult (src/analysis/result.rs:183-216) plus the integer parity views of the C ABI."""

    bpm: float
    bpm_confidence: float
    key: Key
    key_confidence: float
    key_clarity: float
    beat_grid: BeatGrid
    grid_stability: float
    metadata: AnalysisMetadata
    # parity views
    trim_start: int = 0
    trim_end: int = 0
    onsets: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int64))
    hmm_beat_frames: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int32))
    time_sig_beats_per_bar: int = 4
    beats_refined: int = 0
    warnings_mask: int = 0
    flags_mask: int = 0
    error: AnalysisError | None = None  # set instead of raising inside analyze_batch (ItemOut.error)


def _opt(v: int):
    return None if v < 0 else bool(v)


def _arr(ptr, n, dtype):
    if n == 0 or not ptr:
        return np.zeros(0, dtype)
    return np.ctypeslib.as_array(ptr, shape=(n,)).astype(dtype, copy=True)


def _flags(mask: int):
    return [name for bit, name in _FLAG_NAMES.items() if mask & bit]


def _convert(r: StratumResult) -> AnalysisResult:
    L = lib()
    if r.status != OK:
        err = AnalysisError(r.status, r.error.decode(errors="replace"))
        meta = AnalysisMetadata(0.0, 0, 0.0, ALGORITHM_VERSION, 0.0, [], [], [], None, None, None, None)
        return AnalysisResult(0.0, 0.0, Key(False, 0), 0.0, 0.0, BeatGrid(np.zeros(0, np.float32), np.zeros(0, np.float32), np.zeros(0, np.float32)),
                              0.0, meta, error=err)
    wb = C.create_string_buffer(2048)
    L.stratum_b200_warning_strings(C.byref(r), wb, 2048)
    warnings = [w for w in wb.value.decode().split("\n") if w]
    meta = AnalysisMetadata(
        duration_seconds=r.duration_seconds, sample_rate=r.sample_rate, processing_time_ms=r.processing_time_ms,
        algorithm_version=ALGORITHM_VERSION, onset_method_consensus=r.onset_method_consensus,
        methods_used=list(METHODS_USED),  # lib.rs:1604-1608
        flags=_flags(r.flags), confidence_warnings=warnings,
        tempogram_multi_res_triggered=_opt(r.tempogram_multi_res_triggered), tempogram_multi_res_used=_opt(r.tempogram_multi_res_used),
        tempogram_percussive_triggered=_opt(r.tempogram_percussive_triggered), tempogram_percussive_used=_opt(r.tempogram_percussive_used),
        tempogram_candidates=None if r.n_tempogram_candidates < 0 else [
            (c.bpm, c.score, c.fft_norm, c.autocorr_norm, bool(c.selected)) for c in (r.tempogram_candidates[i] for i in range(r.n_tempogram_candidates))])
    grid = BeatGrid(_arr(r.beats, r.n_beats, np.float32), _arr(r.downbeats, r.n_downbeats, np.float32), _arr(r.bars, r.n_bars, np.float32))
    return AnalysisResult(
        bpm=r.bpm, bpm_confidence=r.bpm_confidence, key=Key(bool(r.key_is_minor), int(r.key_index)), key_confidence=r.key_confidence,
        key_clarity=r.key_clarity, beat_grid=grid, grid_stability=r.grid_stability, metadata=meta, trim_start=int(r.trim_start),
        trim_end=int(r.trim_end), onsets=_arr(r.onsets, r.n_onsets, np.int64), hmm_beat_frames=_arr(r.hmm_beat_frames, r.n_hmm_beat_frames, np.int32),
        time_sig_beats_per_bar=int(r.time_sig_beats_per_bar), beats_refined=int(r.beats_refined), warnings_mask=int(r.warnings), flags_mask=int(r.flags))


def _cfg_ptr(config: AnalysisConfig | None):
    return C.byref(config._c) if config is not None else None


def analyze_audio(samples, sample_rate: int, config: AnalysisConfig | None = None) -> AnalysisResult:
    """analyze_audio(&samples, sample_rate, config) -> Result<AnalysisResult, AnalysisError> (src/lib.rs:86-90)."""
    x = np.ascontiguousarray(samples, dtype=np.float32)
    r = StratumResult()
    st = lib().stratum_b200_analyze_audio(x.ctypes.data if x.size else None, x.size, int(sample_rate), _cfg_ptr(config), C.byref(r))
    try:
        if st != OK:
            raise AnalysisError(st, r.error.decode(errors="replace") or last_error())
        return _convert(r)
    finally:
        lib().stratum_b200_result_free(C.byref(r), 1)


def compute_confidence(result: AnalysisResult) -> AnalysisConfidence:
    """compute_confidence(&AnalysisResult) (src/analysis/confidence.rs:121-179)."""
    r = StratumResult()
    r.bpm, r.bpm_confidence = result.bpm, result.bpm_confidence
    r.key_confidence, r.key_clarity, r.grid_stability = result.key_confidence, result.key_clarity, result.grid_stability
    r.warnings, r.flags = result.warnings_mask, result.flags_mask
    out = StratumConfidence()
    lib().stratum_b200_compute_confidence(C.byref(r), C.byref(out))
    return AnalysisConfidence(out.bpm_confidence, out.key_confidence, out.grid_stability, out.overall_confidence, _flags(out.flags))


def _fail(st: int, res, n: int):
    """Batch-level error: results of waves that completed before it own heap arrays — release them, then raise."""
    msg = last_error()
    lib().stratum_b200_result_free(res, n)
    raise AnalysisError(st, msg)


def _collect(res, n) -> list:
    try:
        return [_convert(res[i]) for i in range(n)]
    finally:
        lib().stratum_b200_result_free(res, n)


def analyze_batch(tracks: Sequence, sample_rates: int | Iterable[int], config: AnalysisConfig | None = None,
                  devices: Sequence[int] | None = None) -> list:
    """Batch surface of examples/analyze_batch.rs:260-326: one result per track, a failed track carries
    ``.error`` instead of aborting the batch.  ``tracks`` are HOST arrays; they are sharded by track
    over ``devices`` (default: the current device)."""
    arrs = [np.ascontiguousarray(t, dtype=np.float32).ravel() for t in tracks]
    n = len(arrs)
    if n == 0:
        return []
    srs = [int(sample_rates)] * n if isinstance(sample_rates, (int, np.integer)) else [int(s) for s in sample_rates]
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([a.size for a in arrs], dtype=np.uint64)
    cat = np.concatenate(arrs) if n > 1 else arrs[0]
    return analyze_batch_packed(cat, offsets, srs, config, devices)


def analyze_batch_packed(samples: np.ndarray, offsets: np.ndarray, sample_rates: Sequence[int], config: AnalysisConfig | None = None,
                         devices: Sequence[int] | None = None) -> list:
    """Same as analyze_batch with the tracks already concatenated (track i = samples[offsets[i]:offsets[i+1]])."""
    samples = np.ascontiguousarray(samples, dtype=np.float32)
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = offsets.size - 1
    srs = np.ascontiguousarray(sample_rates, dtype=np.uint32)
    res = (StratumResult * n)()
    dev = (C.c_int32 * len(devices))(*devices) if devices else None
    st = lib().stratum_b200_analyze_batch(samples.ctypes.data if samples.size else None, offsets.ctypes.data_as(C.POINTER(C.c_uint64)),
                                          srs.ctypes.data_as(C.POINTER(_u)), n, _cfg_ptr(config), dev, len(devices) if devices else 0, res)
    if st != OK:
        _fail(st, res, n)
    return _collect(res, n)


def analyze_batch_pcm16(tracks: Sequence, sample_rates: int | Iterable[int], config: AnalysisConfig | None = None,
                        devices: Sequence[int] | None = None) -> list:
    """Decoder-side batch entry (SURVEY §8f n4): ``tracks`` are int16 PCM arrays, shape (frames,) for mono or
    (frames, channels) interleaved.  The PCM is uploaded as is (half the PCIe bytes of f32) and converted on the device
    with the reference decoder's arithmetic (examples/analyze_batch.rs:96-113)."""
    arrs = [np.ascontiguousarray(t, dtype=np.int16) for t in tracks]
    n = len(arrs)
    if n == 0:
        return []
    chans = np.array([a.shape[1] if a.ndim == 2 else 1 for a in arrs], dtype=np.uint32)
    flat = [a.reshape(-1) for a in arrs]
    srs = np.ascontiguousarray([int(sample_rates)] * n if isinstance(sample_rates, (int, np.integer)) else [int(s) for s in sample_rates], dtype=np.uint32)
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([a.size for a in flat], dtype=np.uint64)
    cat = np.concatenate(flat) if n > 1 else flat[0]
    res = (StratumResult * n)()
    dev = (C.c_int32 * len(devices))(*devices) if devices else None
    st = lib().stratum_b200_analyze_batch_pcm16(cat.ctypes.data if cat.size else None, offsets.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                srs.ctypes.data_as(C.POINTER(_u)), chans.ctypes.data_as(C.POINTER(_u)), n, _cfg_ptr(config), dev,
                                                len(devices) if devices else 0, res)
    if st != OK:
        _fail(st, res, n)
    return _collect(res, n)


PCM_U8, PCM_S16, PCM_S24, PCM_S32, PCM_F32, PCM_F64 = 1, 2, 3, 4, 5, 6  # StratumPcmFormat
_PCM_BYTES = {PCM_U8: 1, PCM_S16: 2, PCM_S24: 3, PCM_S32: 4, PCM_F32: 4, PCM_F64: 8}


@dataclass
class PcmTrack:
    """Undecoded interleaved PCM of one track: ``data`` = the bytes of the sample frames (little-endian, 24-bit packed)."""

    data: np.ndarray  # uint8
    fmt: int          # PCM_*
    channels: int
    sample_rate: int

    @property
    def frames(self) -> int:
        return self.data.size // (_PCM_BYTES[self.fmt] * self.channels)


def read_wav(path) -> PcmTrack:
    """RIFF/WAVE container -> PcmTrack without touching the samples: WAVE_FORMAT_PCM (8/16/24/32 bit), WAVE_FORMAT_IEEE_FLOAT
    (32/64 bit) and WAVE_FORMAT_EXTENSIBLE with a PCM or IEEE-float sub-format, any channel count (the formats symphonia's WAV
    reader hands to the reference's decoder loop, examples/analyze_batch.rs:30-178).  Conversion and mixdown happen on the device."""
    import struct

    raw = np.fromfile(str(path), dtype=np.uint8)
    b = raw.tobytes() if raw.size < (1 << 16) else None
    hdr = bytes(raw[:12])
    if len(hdr) < 12 or hdr[:4] != b"RIFF" or hdr[8:12] != b"WAVE":
        raise ValueError("not a RIFF/WAVE file")
    pos, fmt, data = 12, None, None
    while pos + 8 <= raw.size:
        cid = bytes(raw[pos:pos + 4])
        (size,) = struct.unpack("<I", bytes(raw[pos + 4:pos + 8]))
        body = pos + 8
        if cid == b"fmt ":
            f = bytes(raw[body:body + min(size, 40)])
            tag, ch, sr, _br, _align, bits = struct.unpack("<HHIIHH", f[:16])
            if tag == 0xFFFE and len(f) >= 40:  # WAVE_FORMAT_EXTENSIBLE: the sub-format GUID starts with the real tag
                (tag,) = struct.unpack("<H", f[24:26])
            fmt = (tag, ch, sr, bits)
        elif cid == b"data":
            end = min(body + size, raw.size)  # a streamed file may carry a bogus length
            data = raw[body:end]
            if fmt is not None:
                break
        pos = body + size + (size & 1)
    del b
    if fmt is None or data is None:
        raise ValueError("WAVE file without fmt/data chunk")
    tag, ch, sr, bits = fmt
    if tag == 1 and bits in (8, 16, 24, 32):
        pf = {8: PCM_U8, 16: PCM_S16, 24: PCM_S24, 32: PCM_S32}[bits]
    elif tag == 3 and bits in (32, 64):
        pf = PCM_F32 if bits == 32 else PCM_F64
    else:
        raise ValueError(f"Unsupported sample format (format tag {tag}, {bits} bit)")
    if ch == 0:
        raise ValueError("WAVE file with zero channels")
    frame = _PCM_BYTES[pf] * ch
    return PcmTrack(np.ascontiguousarray(data[: data.size // frame * frame]), pf, ch, sr)


def analyze_batch_pcm(tracks: Sequence[PcmTrack], config: AnalysisConfig | None = None, devices: Sequence[int] | None = None) -> list:
    """stratum_b200_analyze_batch_pcm: undecoded PCM tracks of any supported format / channel count in one call."""
    n = len(tracks)
    if n == 0:
        return []
    flat = [np.ascontiguousarray(t.data, dtype=np.uint8).reshape(-1) for t in tracks]
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([a.size for a in flat], dtype=np.uint64)
    cat = np.concatenate(flat) if n > 1 else flat[0]
    srs = np.ascontiguousarray([t.sample_rate for t in tracks], dtype=np.uint32)
    chans = np.ascontiguousarray([t.channels for t in tracks], dtype=np.uint32)
    fmts = np.ascontiguousarray([t.fmt for t in tracks], dtype=np.uint32)
    res = (StratumResult * n)()
    dev = (C.c_int32 * len(devices))(*devices) if devices else None
    L = lib()
    L.stratum_b200_analyze_batch_pcm.argtypes = [C.c_void_p, C.POINTER(C.c_uint64), C.POINTER(_u), C.POINTER(_u), C.POINTER(_u), C.c_uint32, C.c_void_p,
                                                 C.POINTER(C.c_int32), C.c_uint32, C.POINTER(StratumResult)]
    cfgp = C.cast(C.byref(config._c), C.c_void_p) if config is not None else None
    st = L.stratum_b200_analyze_batch_pcm(cat.ctypes.data if cat.size else None, offsets.ctypes.data_as(C.POINTER(C.c_uint64)), srs.ctypes.data_as(C.POINTER(_u)),
                                          chans.ctypes.data_as(C.POINTER(_u)), fmts.ctypes.data_as(C.POINTER(_u)), n, cfgp, dev, len(devices) if devices else 0, res)
    if st != OK:
        _fail(st, res, n)
    return _collect(res, n)


@dataclass
class Loudness:
    """ITU-R BS.1770-4 / EBU R128 loudness of one track or album (include/stratum_b200.h: StratumLoudness).  Loudness values are in LUFS,
    the range in LU, peaks linear (full scale 1.0); undefined loudness values are ``float("-inf")``."""

    integrated_lufs: float
    momentary_max_lufs: float
    short_term_max_lufs: float
    loudness_range_lu: float
    sample_peak: float
    true_peak: float
    n_momentary: int
    n_short_term: int
    sample_rate: int
    channels: int
    frames: int
    error: AnalysisError | None = None  # set instead of raising for a track that failed on its own


def _loudness(r: StratumLoudness) -> Loudness:
    err = AnalysisError(r.status, r.error.decode(errors="replace")) if r.status != OK else None
    return Loudness(r.integrated_lufs, r.momentary_max_lufs, r.short_term_max_lufs, r.loudness_range_lu, r.sample_peak, r.true_peak,
                    int(r.n_momentary), int(r.n_short_term), int(r.sample_rate), int(r.channels), int(r.frames), err)


def _pcm_tables(tracks: Sequence[PcmTrack]):
    n = len(tracks)
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum([t.data.size for t in tracks], dtype=np.uint64)
    srs = np.ascontiguousarray([t.sample_rate for t in tracks], dtype=np.uint32)
    chans = np.ascontiguousarray([t.channels for t in tracks], dtype=np.uint32)
    fmts = np.ascontiguousarray([t.fmt for t in tracks], dtype=np.uint32)
    return offsets, srs, chans, fmts


def loudness_batch_pcm(tracks: Sequence[PcmTrack], devices: Sequence[int] | None = None) -> list:
    """stratum_b200_loudness_batch_pcm: integrated loudness, maxima, loudness range and peaks of undecoded PCM tracks, measured on
    the device and sharded over ``devices`` (default: the current device).  A failed track carries ``.error``."""
    n = len(tracks)
    if n == 0:
        return []
    flat = [np.ascontiguousarray(t.data, dtype=np.uint8).reshape(-1) for t in tracks]
    cat = np.concatenate(flat) if n > 1 else flat[0]
    offsets, srs, chans, fmts = _pcm_tables(tracks)
    res = (StratumLoudness * n)()
    dev = (C.c_int32 * len(devices))(*devices) if devices else None
    st = lib().stratum_b200_loudness_batch_pcm(cat.ctypes.data if cat.size else None, offsets.ctypes.data_as(C.POINTER(C.c_uint64)),
                                               srs.ctypes.data_as(C.POINTER(_u)), chans.ctypes.data_as(C.POINTER(_u)), fmts.ctypes.data_as(C.POINTER(_u)),
                                               n, dev, len(devices) if devices else 0, res)
    if st != OK:
        _raise(st)
    return [_loudness(res[i]) for i in range(n)]


def loudness_batch_pcm_device(d_pcm_ptr: int, byte_offsets: np.ndarray, sample_rates: Sequence[int], channels: Sequence[int], formats: Sequence[int],
                              device: int = -1) -> list:
    """stratum_b200_loudness_batch_pcm_device: the same with the PCM already in device memory (``d_pcm_ptr`` = device address of the
    concatenated track bytes, e.g. ``tensor.data_ptr()``; track i = bytes [byte_offsets[i], byte_offsets[i + 1]))."""
    offsets = np.ascontiguousarray(byte_offsets, dtype=np.uint64)
    n = offsets.size - 1
    srs = np.ascontiguousarray(sample_rates, dtype=np.uint32)
    chans = np.ascontiguousarray(channels, dtype=np.uint32)
    fmts = np.ascontiguousarray(formats, dtype=np.uint32)
    if not (srs.size == chans.size == fmts.size == n):
        raise ValueError("one sample rate, channel count and format per track")
    res = (StratumLoudness * max(n, 1))()
    st = lib().stratum_b200_loudness_batch_pcm_device(C.c_void_p(d_pcm_ptr), offsets.ctypes.data_as(C.POINTER(C.c_uint64)), srs.ctypes.data_as(C.POINTER(_u)),
                                                      chans.ctypes.data_as(C.POINTER(_u)), fmts.ctypes.data_as(C.POINTER(_u)), n, device, res)
    if st != OK:
        _raise(st)
    return [_loudness(res[i]) for i in range(n)]


NO_ALBUM = 0xFFFFFFFF  # STRATUM_NO_ALBUM


def _album_ids(albums: Sequence[int | None], n_tracks: int, n_albums: int | None):
    if len(albums) != n_tracks:
        raise ValueError("one album id (or None) per track")
    if any(a is not None and (int(a) < 0 or int(a) >= NO_ALBUM) for a in albums):
        raise ValueError("album ids are non-negative integers below 0xFFFFFFFF, or None")
    ids = np.ascontiguousarray([NO_ALBUM if a is None else int(a) for a in albums], dtype=np.uint32).reshape(-1)
    if n_albums is None:
        n_albums = max((int(a) + 1 for a in albums if a is not None), default=0)
    return ids, int(n_albums)


def loudness_albums_pcm(tracks: Sequence[PcmTrack], albums: Sequence[int | None], n_albums: int | None = None,
                        devices: Sequence[int] | None = None) -> tuple:
    """stratum_b200_loudness_albums_pcm: the per-track results of ``loudness_batch_pcm`` and the loudness of albums (ReplayGain /
    R128 album values), each measured over the pooled 400 ms blocks and 3 s windows of its members.  ``albums[i]`` is the album id of
    track i (``None``: no album); ``n_albums`` defaults to the largest id + 1.  Returns ``(tracks, albums)``, two lists of
    ``Loudness``; an album with a failed member, or one that no track names, carries ``.error``."""
    n = len(tracks)
    ids, na = _album_ids(albums, n, n_albums)
    flat = [np.ascontiguousarray(t.data, dtype=np.uint8).reshape(-1) for t in tracks]
    cat = np.concatenate(flat) if n > 1 else (flat[0] if n else np.zeros(0, np.uint8))
    offsets, srs, chans, fmts = _pcm_tables(tracks)
    res = (StratumLoudness * max(n, 1))()
    alb = (StratumLoudness * max(na, 1))()
    dev = (C.c_int32 * len(devices))(*devices) if devices else None
    st = lib().stratum_b200_loudness_albums_pcm(cat.ctypes.data if cat.size else None, offsets.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                srs.ctypes.data_as(C.POINTER(_u)), chans.ctypes.data_as(C.POINTER(_u)), fmts.ctypes.data_as(C.POINTER(_u)),
                                                n, ids.ctypes.data_as(C.POINTER(_u)), na, dev, len(devices) if devices else 0, res, alb)
    if st != OK:
        _raise(st)
    return [_loudness(res[i]) for i in range(n)], [_loudness(alb[a]) for a in range(na)]


def loudness_albums_pcm_device(d_pcm_ptr: int, byte_offsets: np.ndarray, sample_rates: Sequence[int], channels: Sequence[int], formats: Sequence[int],
                               albums: Sequence[int | None], n_albums: int | None = None, device: int = -1) -> tuple:
    """stratum_b200_loudness_albums_pcm_device: ``loudness_albums_pcm`` with the PCM already in device memory (arguments as
    ``loudness_batch_pcm_device``)."""
    offsets = np.ascontiguousarray(byte_offsets, dtype=np.uint64)
    n = offsets.size - 1
    srs = np.ascontiguousarray(sample_rates, dtype=np.uint32)
    chans = np.ascontiguousarray(channels, dtype=np.uint32)
    fmts = np.ascontiguousarray(formats, dtype=np.uint32)
    if not (srs.size == chans.size == fmts.size == n):
        raise ValueError("one sample rate, channel count and format per track")
    ids, na = _album_ids(albums, n, n_albums)
    res = (StratumLoudness * max(n, 1))()
    alb = (StratumLoudness * max(na, 1))()
    st = lib().stratum_b200_loudness_albums_pcm_device(C.c_void_p(d_pcm_ptr), offsets.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                       srs.ctypes.data_as(C.POINTER(_u)), chans.ctypes.data_as(C.POINTER(_u)),
                                                       fmts.ctypes.data_as(C.POINTER(_u)), n, ids.ctypes.data_as(C.POINTER(_u)), na, device, res, alb)
    if st != OK:
        _raise(st)
    return [_loudness(res[i]) for i in range(n)], [_loudness(alb[a]) for a in range(na)]


def analyze_loudness_pcm(tracks: Sequence[PcmTrack], config: AnalysisConfig | None = None, albums: Sequence[int | None] | None = None,
                         n_albums: int | None = None, devices: Sequence[int] | None = None) -> tuple:
    """stratum_b200_analyze_loudness_pcm: ``analyze_batch_pcm`` and ``loudness_albums_pcm`` of the same tracks from one upload.
    Returns ``(results, loudness, album_loudness)``: the analysis results as ``analyze_batch_pcm`` returns them, one ``Loudness`` per
    track and one per album (``[]`` without ``albums``).  A track's analysis and its loudness fail or succeed independently."""
    n = len(tracks)
    if albums is None:
        if n_albums:
            raise ValueError("n_albums without album ids")
        ids, na = None, 0
    else:
        ids, na = _album_ids(albums, n, n_albums)
    flat = [np.ascontiguousarray(t.data, dtype=np.uint8).reshape(-1) for t in tracks]
    cat = np.concatenate(flat) if n > 1 else (flat[0] if n else np.zeros(0, np.uint8))
    offsets, srs, chans, fmts = _pcm_tables(tracks)
    res = (StratumResult * max(n, 1))()
    loud = (StratumLoudness * max(n, 1))()
    alb = (StratumLoudness * max(na, 1))()
    dev = (C.c_int32 * len(devices))(*devices) if devices else None
    cfgp = C.cast(C.byref(config._c), C.c_void_p) if config is not None else None
    st = lib().stratum_b200_analyze_loudness_pcm(cat.ctypes.data if cat.size else None, offsets.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                 srs.ctypes.data_as(C.POINTER(_u)), chans.ctypes.data_as(C.POINTER(_u)), fmts.ctypes.data_as(C.POINTER(_u)),
                                                 n, cfgp, ids.ctypes.data_as(C.POINTER(_u)) if ids is not None else None, na, dev,
                                                 len(devices) if devices else 0, res, loud, alb)
    if st != OK:
        _fail(st, res, n)
    return _collect(res, n), [_loudness(loud[i]) for i in range(n)], [_loudness(alb[a]) for a in range(na)]


def loudness_filters(sample_rate: int) -> tuple:
    """The host-side filters of the loudness measurement: (K-weighting coefficients [b0 b1 b2 a1 a2] x 2 stages in float64,
    true-peak taps in float32, oversampling factor).  Raises for a sample rate outside 8000..384000 Hz."""
    k = np.zeros(10, np.float64)
    t = np.zeros(49, np.float32)
    L = lib().stratum_b200_debug_loudness_filters(int(sample_rate), k.ctypes.data_as(C.POINTER(C.c_double)), t.ctypes.data_as(C.POINTER(_f)))
    if L < 0:
        raise AnalysisError(4, f"sample rate {sample_rate} Hz is outside 8000..384000 Hz")
    return k, t, L


def analyze_batch_device(d_samples_ptr: int, offsets: np.ndarray, sample_rates: Sequence[int], config: AnalysisConfig | None = None,
                         device: int = -1, convert: bool = True):
    """Batch already resident in device memory (``d_samples_ptr`` = device address of the concatenated f32
    samples, e.g. ``tensor.data_ptr()``).  With ``convert=False`` returns the raw ctypes result array and
    the caller must pass it to ``free_results``."""
    offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
    n = offsets.size - 1
    srs = np.ascontiguousarray(sample_rates, dtype=np.uint32)
    res = (StratumResult * n)()
    st = lib().stratum_b200_analyze_batch_device(C.c_void_p(d_samples_ptr), offsets.ctypes.data_as(C.POINTER(C.c_uint64)),
                                                 srs.ctypes.data_as(C.POINTER(_u)), n, _cfg_ptr(config), device, res)
    if st != OK:
        _fail(st, res, n)
    if not convert:
        return res
    return _collect(res, n)


def shard_bounds(n_tracks: int, shard: int, n_shards: int) -> tuple:
    """Contiguous shard [a, b) of a batch for device/rank ``shard`` — the rule stratum_b200_analyze_batch uses
    across ``device_ids`` (csrc/engine.cu) and bench.py uses across ranks: tracks are independent
    (examples/analyze_batch.rs:260-326), so sharding by track needs no data-path collective."""
    return (n_tracks * shard) // n_shards, (n_tracks * (shard + 1)) // n_shards


def free_results(res) -> None:
    lib().stratum_b200_result_free(res, len(res))


# ---- stage-level helpers (parity tests, bench instrumentation) ---------------------------------------
def stft(samples, frame_size: int, hop: int, gain: float = 1.0) -> np.ndarray:
    """compute_stft (src/features/chroma/extractor.rs:301-359) on the device."""
    x = np.ascontiguousarray(samples, dtype=np.float32)
    if x.size < frame_size:
        return np.zeros((0, frame_size // 2 + 1), np.float32)
    nf = (x.size - frame_size) // hop + 1
    out = np.zeros((nf, frame_size // 2 + 1), dtype=np.float32)
    got = lib().stratum_b200_stft(x.ctypes.data, x.size, frame_size, hop, gain, out.ctypes.data, out.size)
    if got < 0:
        _raise(int(-got))
    assert got == nf
    return out


def synth_batch(d_out_ptr: int, n_tracks: int, n_samples: int, sample_rate: int, params5: np.ndarray, device: int = -1) -> None:
    p = np.ascontiguousarray(params5, dtype=np.float32).reshape(n_tracks, 5)
    st = lib().stratum_b200_synth_batch(C.c_void_p(d_out_ptr), n_tracks, n_samples, sample_rate, p.ctypes.data_as(C.POINTER(_f)), device)
    if st != OK:
        _raise(st)


def debug_enable(on: bool) -> None:
    lib().stratum_b200_debug_enable(int(on))


def debug_array(name: str) -> np.ndarray | None:
    n = lib().stratum_b200_debug_array(name.encode(), None, 0)
    if n < 0:
        return None
    out = np.zeros(n, dtype=np.float32)
    if n:
        lib().stratum_b200_debug_array(name.encode(), out.ctypes.data, n)
    return out


def stage_timing(on: bool) -> None:
    lib().stratum_b200_stage_timing_enable(int(on))


def stage_times(reset: bool = False) -> dict:
    names = C.create_string_buffer(4096)
    ms = (C.c_double * 64)()
    n = lib().stratum_b200_stage_times(names, 4096, ms, 64)
    out = {nm: ms[i] for i, nm in enumerate([s for s in names.value.decode().split("\n") if s][:n])}
    if reset:
        lib().stratum_b200_stage_times_reset()
    return out


def last_call_device_ms() -> float:
    return float(lib().stratum_b200_last_call_device_ms())


def last_call_waves() -> int:
    return int(lib().stratum_b200_last_call_waves())


def transfer_bytes() -> tuple:
    a, b = C.c_uint64(), C.c_uint64()
    lib().stratum_b200_transfer_bytes(C.byref(a), C.byref(b))
    return int(a.value), int(b.value)


def launch_count() -> int:
    return int(lib().stratum_b200_launch_count())


def device_count() -> int:
    return int(lib().stratum_b200_device_count())


def shutdown() -> None:
    lib().stratum_b200_shutdown()
