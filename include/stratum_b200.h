/*
 * stratum_b200.h — C ABI of the B200-native replacement for stratum-dsp's per-track analysis
 * hot path.  Every entry point is plain C (pointers + sizes, no C++ or torch types) so the
 * reference's Rust crate can bind it through a thin `-sys` FFI crate (INTEGRATION.md shows the
 * binding).  All `file:line` citations are relative to the reference repository.
 *
 *   analyze_audio(&[f32], u32, AnalysisConfig) -> Result<AnalysisResult, AnalysisError>
 *                                                    src/lib.rs:86-90      -> stratum_b200_analyze_audio
 *   paths.par_iter().map(analyze_audio + compute_confidence)
 *                                                    examples/analyze_batch.rs:260-326 -> stratum_b200_analyze_batch
 *   compute_confidence(&AnalysisResult)              src/analysis/confidence.rs:121  -> stratum_b200_compute_confidence
 *   AnalysisConfig::default()                        src/config.rs:594-744          -> stratum_b200_config_default
 *   AnalysisError                                    src/error.rs:7-22              -> StratumStatus + message
 *   Key::name() / Key::numerical()                   src/analysis/result.rs:31-87   -> stratum_b200_key_name
 *
 * There is no CPU fallback: every compute entry point fails with STRATUM_PROCESSING_ERROR when
 * no CUDA device is usable.
 */
#ifndef STRATUM_B200_H
#define STRATUM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STRATUM_B200_ABI_VERSION 2

/* AnalysisError variants (src/error.rs:7-22); 0 = Ok. */
typedef enum StratumStatus {
    STRATUM_OK = 0,
    STRATUM_INVALID_INPUT = 1,
    STRATUM_DECODING_ERROR = 2,
    STRATUM_PROCESSING_ERROR = 3,
    STRATUM_NOT_IMPLEMENTED = 4,
    STRATUM_NUMERICAL_ERROR = 5
} StratumStatus;

/* NormalizationMethod (src/preprocessing/normalization.rs:29-37). */
enum { STRATUM_NORM_PEAK = 0, STRATUM_NORM_RMS = 1, STRATUM_NORM_LOUDNESS = 2 };

/* confidence_warnings (src/lib.rs:1567-1589) as a bitmask; stratum_b200_warning_strings rebuilds the
 * exact strings compute_confidence matches on. */
enum {
    STRATUM_WARN_BPM_FAILED = 1,
    STRATUM_WARN_LOW_GRID_STABILITY = 2,
    STRATUM_WARN_LOW_KEY_CONFIDENCE = 4,
    STRATUM_WARN_LOW_KEY_CLARITY = 8
};
/* AnalysisFlag (src/analysis/result.rs:157-167). */
enum { STRATUM_FLAG_MULTIMODAL_BPM = 1, STRATUM_FLAG_WEAK_TONALITY = 2, STRATUM_FLAG_TEMPO_VARIATION = 4, STRATUM_FLAG_ONSET_AMBIGUOUS = 8 };

/* AnalysisConfig (src/config.rs:8-592).  Fields keep the reference's names.  Switches whose
 * non-default branch is not built yet are validated by the library: a value that would select
 * such a branch is rejected with STRATUM_NOT_IMPLEMENTED instead of being silently ignored. */
typedef struct StratumConfig {
    uint32_t abi_version; /* = STRATUM_B200_ABI_VERSION */
    float min_amplitude_db;
    int32_t normalization; /* STRATUM_NORM_* */
    int32_t enable_normalization;
    int32_t enable_silence_trimming;
    int32_t enable_onset_consensus;
    float onset_threshold_percentile;
    uint32_t onset_consensus_tolerance_ms;
    float onset_consensus_weights[4];
    int32_t enable_hpss_onsets;
    int32_t force_legacy_bpm;
    int32_t enable_bpm_fusion;
    int32_t enable_legacy_bpm_guardrails;
    int32_t enable_tempogram_multi_resolution;
    uint32_t tempogram_multi_res_top_k;
    float tempogram_multi_res_w512, tempogram_multi_res_w256, tempogram_multi_res_w1024;
    float tempogram_multi_res_structural_discount;
    float tempogram_multi_res_double_time_512_factor;
    float tempogram_multi_res_margin_threshold;
    int32_t tempogram_multi_res_use_human_prior;
    int32_t enable_tempogram_percussive_fallback;
    int32_t enable_tempogram_band_fusion;
    float tempogram_band_low_max_hz, tempogram_band_mid_max_hz, tempogram_band_high_max_hz;
    float tempogram_band_w_full, tempogram_band_w_low, tempogram_band_w_mid, tempogram_band_w_high;
    int32_t tempogram_band_seed_only;
    float tempogram_band_support_threshold, tempogram_band_consensus_bonus;
    float tempogram_novelty_w_spectral, tempogram_novelty_w_energy, tempogram_novelty_w_hfc;
    uint32_t tempogram_novelty_local_mean_window, tempogram_novelty_smooth_window;
    int32_t enable_tempogram_mel_novelty;
    uint32_t tempogram_mel_n_mels;
    float tempogram_mel_fmin_hz, tempogram_mel_fmax_hz;
    uint32_t tempogram_mel_max_filter_bins;
    float tempogram_mel_weight;
    uint32_t tempogram_superflux_max_filter_bins;
    int32_t emit_tempogram_candidates;
    uint32_t tempogram_candidates_top_n;
    float legacy_bpm_preferred_min, legacy_bpm_preferred_max, legacy_bpm_soft_min, legacy_bpm_soft_max;
    float legacy_bpm_conf_mul_preferred, legacy_bpm_conf_mul_soft, legacy_bpm_conf_mul_extreme;
    float min_bpm, max_bpm, bpm_resolution;
    uint32_t frame_size, hop_size;
    float soft_mapping_sigma;
    uint32_t key_spectrogram_smooth_margin;
    int32_t enable_key_frame_weighting;
    float key_min_tonalness, key_tonalness_power, key_energy_power;
    int32_t enable_key_harmonic_mask;
    float key_harmonic_mask_power;
    int32_t enable_key_stft_override;
    uint32_t key_stft_frame_size, key_stft_hop_size;
    int32_t enable_key_segment_voting;
    uint32_t key_segment_len_frames, key_segment_hop_frames;
    float key_segment_min_clarity;
    int32_t enable_key_hpcp;
    uint32_t key_hpcp_peaks_per_frame, key_hpcp_num_harmonics;
    float key_hpcp_harmonic_decay, key_hpcp_mag_power;
    /* optional key-path variants (SURVEY §8a a39; all off by default, config.rs:683-741); their parameters follow below */
    int32_t enable_key_hpss_harmonic, enable_key_log_frequency, enable_key_beat_synchronous, enable_key_multi_scale,
        enable_key_ensemble, enable_key_median, enable_key_tuning_compensation, enable_key_edge_trim, enable_key_mode_heuristic,
        enable_key_hpcp_whitening, enable_key_hpcp_bass_blend, enable_key_minor_harmonic_bonus;
    float chroma_sharpening_power; /* > 1 sharpens the chroma vectors (chroma/normalization.rs:41-65) */
    uint32_t hpss_margin;          /* median half-width of the HPSS filters (config.rs:43, default 10; at most 10 here) */
    int32_t soft_chroma_mapping;   /* chroma folding (enable_key_hpcp = 0): Gaussian soft mapping (config.rs:244, default 1) */
    int32_t enable_key_spectrogram_time_smoothing; /* used when the harmonic mask is off (config.rs:261, default 1) */
    /* parameters of the optional key-path variants (config.rs:683-741) */
    int32_t key_template_set;              /* TemplateSet (key/templates.rs:16-22): 0 = KrumhanslKessler, 1 = Temperley */
    float key_edge_trim_fraction;
    float key_mode_third_ratio_margin, key_mode_flip_min_score_ratio;
    float key_minor_leading_tone_bonus_weight;
    float key_ensemble_kk_weight, key_ensemble_temperley_weight;
    uint32_t key_multi_scale_n_lengths;    /* Vec<usize> key_multi_scale_lengths as count + fixed array (at most 8 scales) */
    uint32_t key_multi_scale_lengths[8];
    uint32_t key_multi_scale_hop;
    float key_multi_scale_min_clarity;
    uint32_t key_multi_scale_n_weights;    /* Vec<f32> key_multi_scale_weights; 0 = empty = equal weights */
    float key_multi_scale_weights[8];
    uint32_t key_median_segment_length_frames, key_median_segment_hop_frames, key_median_min_segments; /* carried, unused: analyze_audio never reads them */
    float key_tuning_max_abs_semitones;
    uint32_t key_tuning_frame_step;
    float key_tuning_peak_rel_threshold;
    uint32_t key_hpss_frame_step, key_hpss_time_margin, key_hpss_freq_margin;
    float key_hpss_mask_power;
    uint32_t key_hpcp_whitening_smooth_bins;
    float key_hpcp_bass_fmin_hz, key_hpcp_bass_fmax_hz, key_hpcp_bass_weight;
} StratumConfig;

/* TempoCandidateDebug (src/analysis/result.rs:170-181). */
typedef struct StratumTempoCandidate {
    float bpm, score, fft_norm, autocorr_norm;
    int32_t selected;
} StratumTempoCandidate;

/* AnalysisResult + AnalysisMetadata (src/analysis/result.rs:183-263; built at src/lib.rs:1592-1619). */
typedef struct StratumResult {
    int32_t status;     /* StratumStatus for this track; a failed track never aborts the batch */
    char error[128];    /* AnalysisError message */
    float bpm, bpm_confidence;
    int32_t key_is_minor; /* Key::Major(i) -> 0, Key::Minor(i) -> 1 */
    uint32_t key_index;   /* 0 = C ... 11 = B */
    float key_confidence, key_clarity;
    float grid_stability;
    /* BeatGrid: seconds; arrays owned by the library, released by stratum_b200_result_free */
    float* beats;
    float* downbeats;
    float* bars;
    uint32_t n_beats, n_downbeats, n_bars;
    /* metadata */
    float duration_seconds;
    uint32_t sample_rate;
    float processing_time_ms;      /* device time of the batch divided by its track count */
    float onset_method_consensus;
    uint32_t warnings;             /* STRATUM_WARN_* */
    uint32_t flags;                /* STRATUM_FLAG_* */
    int32_t tempogram_multi_res_triggered, tempogram_multi_res_used;       /* Option<bool>: -1 = None */
    int32_t tempogram_percussive_triggered, tempogram_percussive_used;
    /* integer views for parity checks (not in the reference struct) */
    uint64_t trim_start, trim_end; /* sample range kept by detect_and_trim */
    int64_t* onsets;               /* consensus onsets handed to the beat tracker (samples) */
    uint32_t n_onsets;
    int32_t* hmm_beat_frames;      /* frame indices t kept by the first HMM pass (hmm.rs:402-435) */
    uint32_t n_hmm_beat_frames;
    int32_t time_sig_beats_per_bar;
    int32_t beats_refined;         /* 1 when the per-segment Bayesian refinement replaced the grid */
    /* metadata.tempogram_candidates: Option<Vec<..>> — n = -1 is None (emit_tempogram_candidates off or tempogram failed) */
    StratumTempoCandidate* tempogram_candidates;
    int32_t n_tempogram_candidates;
} StratumResult;

/* AnalysisConfidence (src/analysis/confidence.rs:32-68). */
typedef struct StratumConfidence {
    float bpm_confidence, key_confidence, grid_stability, overall_confidence;
    uint32_t flags; /* STRATUM_FLAG_* */
} StratumConfidence;

/* AnalysisConfig::default() — src/config.rs:594-744. */
void stratum_b200_config_default(StratumConfig* cfg);

/* analyze_batch surface (examples/analyze_batch.rs:260-326): track i is
 * samples[offsets[i] .. offsets[i+1]) at sample_rates[i]; `samples` is a HOST pointer (pinned or
 * pageable).  Tracks are sharded across `device_ids[0..n_devices)` (NULL/0 = current device);
 * results are gathered on the host.  Returns STRATUM_OK when the batch ran (per-track outcomes
 * are in out[i].status) or an error when nothing could run (bad arguments, no CUDA device). */
int32_t stratum_b200_analyze_batch(const float* samples, const uint64_t* offsets, const uint32_t* sample_rates, uint32_t n_tracks,
                                   const StratumConfig* cfg, const int32_t* device_ids, uint32_t n_devices, StratumResult* out);

/* Decoder-side entry (SURVEY §8f n4): track i is INTERLEAVED 16-bit PCM with channels[i] channels,
 * pcm[offsets[i] .. offsets[i+1]) (offsets in int16 elements; a multiple of channels[i] per track).  The PCM is
 * uploaded as is — half the PCIe bytes of f32 — and converted on the device exactly like the reference's decoder
 * loop (examples/analyze_batch.rs:96-113): mono `s as f32 / 32768.0`; multi-channel the left-to-right f32 sum of the
 * per-channel values divided by the channel count.  Everything else as stratum_b200_analyze_batch. */
int32_t stratum_b200_analyze_batch_pcm16(const int16_t* pcm, const uint64_t* offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                         uint32_t n_tracks, const StratumConfig* cfg, const int32_t* device_ids, uint32_t n_devices, StratumResult* out);

/* General decoder-side entry: every sample format the reference's decoder loop converts (examples/analyze_batch.rs:70-165).
 * Track i is interleaved PCM in formats[i] (StratumPcmFormat) with channels[i] channels at pcm[byte_offsets[i] .. byte_offsets[i+1])
 * (BYTE offsets; a whole number of frames per track; little-endian; 24-bit samples packed in 3 bytes).  Conversion and mixdown run on
 * the device with the reference's arithmetic: u8 (s - 128) / 128, s16 s / 32768, s24 s / 8388608, s32 s as f32 / 2147483648, f32 as
 * is, f64 as f32; channels summed left to right in f32 from 0.0 and divided by the channel count.  Compressed formats stay on the
 * caller's side (a decoder library's job); what it hands over is PCM in one of these layouts. */
typedef enum StratumPcmFormat {
    STRATUM_PCM_U8 = 1,
    STRATUM_PCM_S16 = 2,
    STRATUM_PCM_S24 = 3,
    STRATUM_PCM_S32 = 4,
    STRATUM_PCM_F32 = 5,
    STRATUM_PCM_F64 = 6
} StratumPcmFormat;
int32_t stratum_b200_analyze_batch_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                       const uint32_t* formats, uint32_t n_tracks, const StratumConfig* cfg, const int32_t* device_ids, uint32_t n_devices,
                                       StratumResult* out);

/* ITU-R BS.1770-4 / EBU R128 loudness of a batch of interleaved PCM tracks (beyond the reference, which has no such output).
 * Track i: `frames` sample frames of C channels at sr Hz, converted to f32 exactly as stratum_b200_analyze_batch_pcm converts them
 * (but never mixed down).  S = (sr + 5) / 10 frames (100 ms).
 *  - Channel weights (libebur128's default map): 1 channel L; 4 channels L R Ls Rs; 5 channels L R C Ls Rs; any other count
 *    0 L, 1 R, 2 C, 3 unused (LFE), 4 Ls, 5 Rs, 6 and up unused.  L, R, C weigh 1.0, Ls and Rs 1.41, unused channels 0.  A caller
 *    whose files state their layout passes a channel map instead (stratum_b200_loudness_mapped_pcm, StratumChannelClass).
 *  - K-weighting: a high shelf (f0 1681.974450955533 Hz, G 3.999843853973347 dB, Q 0.7071752369554196) and a high-pass
 *    (f0 38.13547087602444 Hz, Q 0.5003270373238773) per channel in cascade, zero state at frame 0, coefficients derived per
 *    sample rate from the analog prototype (at 48 kHz they equal BS.1770-4's tables).
 *  - Momentary block j covers frames [jS, jS + 4S), j < J = max(0, floor(frames / S) - 3); short-term window k covers
 *    [kS, kS + 30S), k < K = max(0, floor(frames / S) - 29).  Power = sum over channels of G_c * mean of y_c^2 over the block;
 *    loudness l = -0.691 + 10 log10(power) (power 0: -INFINITY).
 *  - integrated_lufs: mean power of the blocks with l > -70 and l > the relative gate (the loudness of the mean power of the blocks
 *    above -70, minus 10 LU).  momentary_max_lufs / short_term_max_lufs: ungated maxima.  All three -INFINITY when undefined.
 *  - loudness_range_lu (EBU Tech 3342): short-term values above -70 LUFS and above the loudness of their mean power minus 20 LU,
 *    sorted ascending; P(p) = v[floor((n - 1) p + 0.5)]; LRA = P(0.95) - P(0.10), 0 when fewer than two values remain.
 *  - sample_peak: max |x| over channels and frames.  true_peak: max(sample_peak, max |u|) where u is each channel upsampled by
 *    L = 4 (sr < 96 kHz), 2 (sr < 192 kHz) or 1 with the 49 taps c[j] = sinc((j - 24) / L) * 0.5 (1 - cos(2 pi j / 48)), samples
 *    outside the track zero.  Both linear, full scale 1.0.
 * Per-track failures (status/error, the batch carries on): 0 frames or sr = 0 -> STRATUM_INVALID_INPUT; sr outside 8000..384000 Hz
 * -> STRATUM_NOT_IMPLEMENTED.  Calls with a null pointer, an unknown format, channels outside 1..64 or a partial frame are rejected
 * whole (STRATUM_INVALID_INPUT).  Results are bit-identical whatever the batch, the upload chunks and the devices. */
typedef struct StratumLoudness {
    int32_t status; char error[128];
    uint32_t sample_rate, channels; uint64_t frames;
    double integrated_lufs, momentary_max_lufs, short_term_max_lufs;  /* -INFINITY when undefined (see above) */
    double loudness_range_lu;
    double sample_peak, true_peak;                                     /* linear full scale */
    uint32_t n_momentary, n_short_term;                                /* J and K */
} StratumLoudness;

/* Host PCM (layout of stratum_b200_analyze_batch_pcm), sharded over `device_ids` and streamed through the double-buffered upload. */
int32_t stratum_b200_loudness_batch_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                        const uint32_t* formats, uint32_t n_tracks, const int32_t* device_ids, uint32_t n_devices, StratumLoudness* out);
/* Same, with the PCM already resident in the memory of device `device_id`. */
int32_t stratum_b200_loudness_batch_pcm_device(const void* d_pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                               const uint32_t* formats, uint32_t n_tracks, int32_t device_id, StratumLoudness* out);

/* Album loudness (ReplayGain 2.0 / R128 album values): track i belongs to album album_of_track[i] < n_albums, or to none
 * (STRATUM_NO_ALBUM).  An album's pooled momentary list is the concatenation of its members' momentary powers (the blocks defined
 * above, each member at its own sample rate, channel count and format), members in ascending track index; its pooled short-term list
 * likewise.
 *  - integrated_lufs: the per-track rule on the pooled momentary list: absolute gate -70 LUFS, relative gate 10 LU below the
 *    loudness of the mean power of the blocks above -70, loudness of the mean power of the blocks above both gates.  A quiet track
 *    can fall under the album's relative gate although it passes its own.
 *  - momentary_max_lufs / short_term_max_lufs: maxima over the pooled lists (-INFINITY for an empty list).
 *  - loudness_range_lu: the per-track range rule on the pooled short-term list.
 *  - sample_peak / true_peak: maxima over the members.  n_momentary / n_short_term: the pooled counts.  frames: the sum over the
 *    members.  sample_rate, channels: 0.
 * An album of one track has that track's values bit for bit, and album values depend only on the members' samples: not on the
 * other tracks, the order of the albums, the upload chunks, the devices or the entry.
 * Album status: STRATUM_OK when every member is measured; otherwise the status of the lowest-index failed member, the error
 * "track <i>: <member's message>" and no values (no album value over a partial album).  An id no track names: STRATUM_INVALID_INPUT,
 * "album has no tracks".  Neither case touches other albums or any track result.
 * Rejected whole (STRATUM_INVALID_INPUT, before any device work), besides what the per-track entries reject: an id at or above
 * n_albums other than STRATUM_NO_ALBUM; a NULL album_of_track or album_out while n_albums > 0.  album_of_track may be NULL when
 * n_albums = 0, which is stratum_b200_loudness_batch_pcm.  out[i] is the per-track result of stratum_b200_loudness_batch_pcm. */
#define STRATUM_NO_ALBUM 0xFFFFFFFFu
int32_t stratum_b200_loudness_albums_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                         const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                         const int32_t* device_ids, uint32_t n_devices, StratumLoudness* out, StratumLoudness* album_out);
/* Same, with the PCM already resident in the memory of device `device_id`. */
int32_t stratum_b200_loudness_albums_pcm_device(const void* d_pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                                int32_t device_id, StratumLoudness* out, StratumLoudness* album_out);
/* Analysis and loudness of one host PCM batch from a single upload (a library scan that wants BPM, key and beat grid next to the
 * track and album gains moves each byte over the host link once instead of twice).  Arguments as stratum_b200_analyze_batch_pcm
 * (pcm ... cfg, device_ids, n_devices, out) and stratum_b200_loudness_albums_pcm (album_of_track, n_albums, loudness_out = its out,
 * album_out).
 *  - out[i] is what stratum_b200_analyze_batch_pcm gives for the same arguments, every field bit for bit except processing_time_ms
 *    (integer views, beat / onset / HMM arrays and tempogram candidates included); release it with stratum_b200_result_free.
 *  - loudness_out[i] and album_out[a] are what stratum_b200_loudness_albums_pcm gives, bit for bit.
 *  - A track's analysis status and its loudness status are independent: an all-zero track fails the analysis ("Audio is entirely
 *    silent after trimming") and is still measured; a track at 7999 Hz fails the loudness (STRATUM_NOT_IMPLEMENTED) and is analysed
 *    as stratum_b200_analyze_batch_pcm analyses it.
 *  - Rejected whole, before any device work: whatever either entry rejects.  STRATUM_NOT_IMPLEMENTED for a configuration
 *    stratum_b200_analyze_batch_pcm refuses; STRATUM_INVALID_INPUT for a NULL pointer (out and loudness_out included), an unknown
 *    format, channels outside 1..64, a partial frame, an album id at or above n_albums other than STRATUM_NO_ALBUM, or a NULL
 *    album_of_track / album_out while n_albums > 0.  n_albums = 0 with album_of_track = NULL: no albums.  Checked in the order of
 *    stratum_b200_analyze_batch_pcm (NULL pointers, the configuration, the PCM layout), then the album ids: the first failure is
 *    the one returned.
 * Tracks are sharded over `device_ids` and streamed through the double-buffered upload as in the two entries; on each device the
 * loudness passes are queued on a stream of their own, so they need not wait behind the analysis waves (where the analysis already
 * keeps the device busy, they still add their own kernel time: DESIGN §2).  Album gates run on the first device once every shard
 * is done. */
int32_t stratum_b200_analyze_loudness_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                          const uint32_t* formats, uint32_t n_tracks, const StratumConfig* cfg, const uint32_t* album_of_track,
                                          uint32_t n_albums, const int32_t* device_ids, uint32_t n_devices, StratumResult* out,
                                          StratumLoudness* loudness_out, StratumLoudness* album_out);

/* Channel maps and per-channel results.  A channel map gives every channel of a track one class (one uint8_t per channel), and the
 * class gives the channel's weight G_c in the power of the loudness definition above (BS.1770-4):
 *   STRATUM_CH_UNUSED     weight 0     LFE, unassigned or ignored channels;
 *   STRATUM_CH_FRONT      weight 1.0   L, R, C and every position with |azimuth| < 60 deg or > 120 deg, or elevation >= 30 deg;
 *   STRATUM_CH_SURROUND   weight 1.41  |azimuth| 60..120 deg at elevation < 30 deg (5.1 Ls / Rs at +-110 deg, the 7.1 side pair at
 *                                      +-90 deg);
 *   STRATUM_CH_DUAL_MONO  weight 2.0   a mono channel played on two loudspeakers (+3.01 dB; libebur128's EBUR128_DUAL_MONO).
 * The default map of each channel count is written in these classes by stratum_b200_loudness_channel_map(0, C, 0, map), and a map
 * with the default classes gives results bit-identical to no map. */
typedef enum StratumChannelClass {
    STRATUM_CH_UNUSED = 0,
    STRATUM_CH_FRONT = 1,
    STRATUM_CH_SURROUND = 2,
    STRATUM_CH_DUAL_MONO = 3
} StratumChannelClass;
/* stratum_b200_loudness_albums_pcm with two more arguments:
 *  - channel_map: NULL, the default map for every track; otherwise sum of channels[i] classes, track i's from index
 *    sum_{j<i} channels[j] on, in frame order.  The power stays sum over c of G_c * mean(y_c^2), summed in channel order.
 *  - channel_out: NULL, no per-channel results; otherwise sum of channels[i] entries in the same layout.  Entry (i, c) is channel c of
 *    track i measured alone as a one-channel programme of weight 1.0, whatever its class: every loudness value, both peaks,
 *    n_momentary and n_short_term, channels = 1, the track's sample_rate and frames, and the track's status and error.  It equals,
 *    bit for bit, the result of stratum_b200_loudness_batch_pcm for a one-channel track holding exactly that channel's samples in
 *    the same format.
 * out[i].sample_peak / true_peak stay the maxima over all channels, unused ones included (the maxima over channel_out's entries).
 * Albums pool their members' momentary and short-term powers, weighted by the members' maps; there are no per-channel album values.
 * Rejected whole (STRATUM_INVALID_INPUT, before any device work), after every check of stratum_b200_loudness_albums_pcm: a class
 * code above STRATUM_CH_DUAL_MONO.  The four stratum_b200_loudness_*_pcm entries are this entry with channel_map = channel_out =
 * NULL. */
int32_t stratum_b200_loudness_mapped_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                         const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                         const uint8_t* channel_map, const int32_t* device_ids, uint32_t n_devices, StratumLoudness* out,
                                         StratumLoudness* album_out, StratumLoudness* channel_out);
/* Same, with the PCM already resident in the memory of device `device_id`. */
int32_t stratum_b200_loudness_mapped_pcm_device(const void* d_pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                                const uint8_t* channel_map, int32_t device_id, StratumLoudness* out, StratumLoudness* album_out,
                                                StratumLoudness* channel_out);
/* stratum_b200_analyze_loudness_pcm with channel_map and channel_out as in stratum_b200_loudness_mapped_pcm.  The map weighs the
 * loudness only: out[i] stays what stratum_b200_analyze_batch_pcm gives (its mixdown is the equal-weight average).  The map is
 * checked after every other check; stratum_b200_analyze_loudness_pcm is this entry with channel_map = channel_out = NULL. */
int32_t stratum_b200_analyze_loudness_mapped_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                 const uint32_t* formats, uint32_t n_tracks, const StratumConfig* cfg, const uint32_t* album_of_track,
                                                 uint32_t n_albums, const uint8_t* channel_map, const int32_t* device_ids, uint32_t n_devices,
                                                 StratumResult* out, StratumLoudness* loudness_out, StratumLoudness* album_out,
                                                 StratumLoudness* channel_out);
/* The classes of a track's `channels` channels (1..64) from a WAVE_FORMAT_EXTENSIBLE channel mask, into map[0 .. channels); no
 * device work.  Mask 0: the default map of the channel count.  Otherwise channel c takes the c-th lowest set bit of the mask, and
 * channels beyond the set bits are UNUSED.  SPEAKER_LOW_FREQUENCY (0x8) and the bits above SPEAKER_TOP_BACK_RIGHT (0x20000) are
 * UNUSED; SIDE_LEFT / SIDE_RIGHT (0x200, 0x400) SURROUND; BACK_LEFT / BACK_RIGHT (0x10, 0x20) SURROUND when the mask has no side
 * bit (quad, 5.1 with back surrounds: they sit at +-110 deg) and FRONT when it has one (7.1: the rear pair sits at +-135..150 deg);
 * every other position (centre, back centre, front-of-centre, the top positions) FRONT.  dual_mono != 0 makes the class of a
 * one-channel track DUAL_MONO unless it is UNUSED.  Returns STRATUM_OK, or STRATUM_INVALID_INPUT for a NULL map or channels
 * outside 1..64. */
int32_t stratum_b200_loudness_channel_map(uint32_t wave_mask, uint32_t channels, int32_t dual_mono, uint8_t* map);
/* Loudness series: the loudness over time that an EBU Tech 3341 meter shows (and `ffmpeg -af ebur128` logs), and where the peaks
 * lie, at the 100 ms step S of the definitions above.  Per measured track, nseg = ceil(frames / S):
 *  - momentary series, J entries: entry j is the loudness l of momentary block j (frames [jS, jS + 4S)), -INFINITY for power 0.
 *    A meter shows it at time (j + 4) S / sr.
 *  - short-term series, K entries: entry k is the loudness of short-term window k (frames [kS, kS + 30S)), likewise.
 *  - sample-peak series, nseg entries: entry s is max |x| over all channels and frames [sS, min((s + 1) S, frames)).
 *  - true-peak series, nseg entries: entry s is the max over all channels of the sample peak and the |u| of the L - 1 interpolated
 *    phases at those frames (the true_peak definition above, restricted to the segment's frames).
 * The channel map weighs the momentary and short-term series exactly as it weighs the summary; the peak series are unweighted and
 * count unused channels, as sample_peak and true_peak do.  The largest entry of each series equals out[i].momentary_max_lufs,
 * short_term_max_lufs, sample_peak and true_peak bit for bit, so an album's maxima are the maxima over its members' entries.  A
 * track that fails (status != STRATUM_OK) has no entries.  There are no per-channel or album series.
 *
 * The lengths of a track's series (host only, no device work; any pointer may be NULL): J, K and nseg of a track of `frames` frames
 * at sample_rate Hz.  Returns STRATUM_OK, or the status a loudness entry gives that track, with all three counts 0. */
int32_t stratum_b200_loudness_series_lengths(uint32_t sample_rate, uint64_t frames, uint32_t* n_momentary, uint32_t* n_short_term, uint32_t* n_peaks);
/* stratum_b200_loudness_mapped_pcm with the four series.  Each array may be NULL, and then that series is neither produced nor read
 * back; otherwise it holds the sum over the tracks of that series' lengths, track i's entries starting at the sum of the lengths of
 * tracks 0 .. i-1 (the layout of channel_out).  Entries of failed tracks are not written.  Every other result is bit-identical with
 * or without series, and stratum_b200_loudness_mapped_pcm is this entry with four NULLs.  The series add no kernel launch: pass 2
 * keeps the peaks of each (segment, channel) and the gate writes the series, which are read back with the results. */
int32_t stratum_b200_loudness_series_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                         const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                         const uint8_t* channel_map, const int32_t* device_ids, uint32_t n_devices, StratumLoudness* out,
                                         StratumLoudness* album_out, StratumLoudness* channel_out, double* momentary_lufs, double* short_term_lufs,
                                         double* sample_peaks, double* true_peaks);
/* Same, with the PCM already resident in the memory of device `device_id`. */
int32_t stratum_b200_loudness_series_pcm_device(const void* d_pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                const uint32_t* formats, uint32_t n_tracks, const uint32_t* album_of_track, uint32_t n_albums,
                                                const uint8_t* channel_map, int32_t device_id, StratumLoudness* out, StratumLoudness* album_out,
                                                StratumLoudness* channel_out, double* momentary_lufs, double* short_term_lufs, double* sample_peaks,
                                                double* true_peaks);
/* stratum_b200_analyze_loudness_mapped_pcm with the four series as in stratum_b200_loudness_series_pcm. */
int32_t stratum_b200_analyze_loudness_series_pcm(const void* pcm, const uint64_t* byte_offsets, const uint32_t* sample_rates, const uint32_t* channels,
                                                 const uint32_t* formats, uint32_t n_tracks, const StratumConfig* cfg, const uint32_t* album_of_track,
                                                 uint32_t n_albums, const uint8_t* channel_map, const int32_t* device_ids, uint32_t n_devices,
                                                 StratumResult* out, StratumLoudness* loudness_out, StratumLoudness* album_out,
                                                 StratumLoudness* channel_out, double* momentary_lufs, double* short_term_lufs, double* sample_peaks,
                                                 double* true_peaks);
/* Host-side filters of the loudness measurement (no device work): kweight10 = stage 1 b0 b1 b2 a1 a2, stage 2 b0 b1 b2 a1 a2 (either
 * may be NULL), taps49 = the true-peak interpolator as the device uses it (f32).  Returns the oversampling factor L, or -1 for a
 * sample rate outside 8000..384000 Hz. */
int32_t stratum_b200_debug_loudness_filters(uint32_t sample_rate, double* kweight10, float* taps49);

/* Same, with `samples` already resident in the memory of device `device_id` (single device). */
int32_t stratum_b200_analyze_batch_device(const float* d_samples, const uint64_t* offsets, const uint32_t* sample_rates, uint32_t n_tracks,
                                          const StratumConfig* cfg, int32_t device_id, StratumResult* out);

/* analyze_audio (src/lib.rs:86-90) = batch of one. Returns out->status. */
int32_t stratum_b200_analyze_audio(const float* samples, uint64_t n_samples, uint32_t sample_rate, const StratumConfig* cfg,
                                   StratumResult* out);

/* compute_confidence — src/analysis/confidence.rs:121-179 (pure host function). */
void stratum_b200_compute_confidence(const StratumResult* result, StratumConfidence* out);

/* confidence_warnings strings, newline separated, exactly as src/lib.rs:1567-1589. Returns the length. */
int32_t stratum_b200_warning_strings(const StratumResult* result, char* buf, size_t cap);

/* Key::name() (numerical = 0) / Key::numerical() (numerical = 1) — src/analysis/result.rs:31-87. */
int32_t stratum_b200_key_name(int32_t key_is_minor, uint32_t key_index, int32_t numerical, char* buf, size_t cap);

/* Releases the arrays inside `n` results (the structs themselves belong to the caller). */
void stratum_b200_result_free(StratumResult* results, uint32_t n);

/* Last library-level error message of the calling thread. */
int32_t stratum_b200_last_error(char* buf, size_t cap);

/* Number of kernel launches issued by this process so far / CUDA devices visible. */
uint64_t stratum_b200_launch_count(void);
int32_t stratum_b200_device_count(void);

/* Frees the per-process device contexts. */
void stratum_b200_shutdown(void);

/* sizeof(StratumConfig) / sizeof(StratumResult) / sizeof(StratumConfidence) / sizeof(StratumLoudness) for which = 0 / 1 / 2 / 3:
 * lets an FFI binding assert that its mirror of the structs matches this build. */
size_t stratum_b200_sizeof(int32_t which);

/* ---- stage-level entry points (kernel parity tests and bench instrumentation) ------------------ */

/* compute_stft (src/features/chroma/extractor.rs:301-359) on the device: `samples` host pointer,
 * out = frames x (frame_size/2+1) magnitudes on the host.  frame_size: a power of two from 64 to 16 384. */
int64_t stratum_b200_stft(const float* samples, uint64_t n, uint32_t frame_size, uint32_t hop, float gain, float* out, uint64_t out_cap);

/* Device-side synthetic generator (tests/synth.py, SURVEY §8d): fills d_out (device) with n_tracks
 * tracks of n_samples each. params: per track {bpm, tonic, minor, phase_frac, chord_amp}. */
int32_t stratum_b200_synth_batch(float* d_out, uint32_t n_tracks, uint64_t n_samples, uint32_t sample_rate, const float* params5,
                                 int32_t device_id);

/* Named intermediate of the most recent single-track analyze call on this thread (debug builds of
 * the parity tests): copies up to cap floats, returns the available length or -1. */
int64_t stratum_b200_debug_array(const char* name, float* out, int64_t cap);
void stratum_b200_debug_enable(int32_t on);

/* Measured FP32 FMA rate of the device in TFLOP/s (8 independent chains per thread, 2 flops per FMA): the second
 * roofline denominator of bench.py (the path is FP32-bound, SURVEY §8d).  0 when no device is usable. */
double stratum_b200_fp32_peak_tflops(int32_t device_id);

/* Self-check of the range-restricted exact divisions the hot kernels use (csrc/common.cuh) against IEEE division on n random
 * operand tuples drawn from their documented ranges; mismatches3 = {a/25, hp/(hp+rp+eps), x/rowmax} mismatch counts (all 0). */
int32_t stratum_b200_debug_check_divisions(uint64_t n, uint32_t seed, uint64_t* mismatches3);

/* Host-side wave planner on its own (no device work): wave index of every track for an arena budget of budget_gb
 * gigabytes; returns the number of waves.  Lets the packing logic be tested without a GPU. */
uint32_t stratum_b200_debug_plan_waves(const uint64_t* offsets, const uint32_t* sample_rates, uint32_t n_tracks, const StratumConfig* cfg, double budget_gb,
                                       uint32_t* wave_of_track);

/* Host-side schedule of the mel-band fold of the novelty features on its own (no device work; csrc/engine.cu: mel_fold_schedule):
 * mel_off = n_mels + 1 entry offsets (n_mels <= 40), schedule256 = 64 chunk starts, 64 chunk ends, 64 partial-sum positions, 41 band
 * starts (padded to 256).  Lets the chunking be tested without a GPU. */
void stratum_b200_debug_mel_schedule(const int32_t* mel_off, uint32_t n_mels, int32_t* schedule256);

/* Host-side BPM hypothesis grid on its own (no device work; csrc/engine.cu: bpm_grid): the values of the reference's f32 loop
 * `bpm = min_bpm; while bpm <= max_bpm { ..; bpm += bpm_resolution }` (tempogram_autocorr.rs:79-178).  Writes the first
 * min(count, cap) values to out (may be NULL) and returns the count, or -1 for an invalid range or a grid of more than 32768
 * hypotheses (which includes every grid whose accumulation stalls).  Such grids are rejected with STRATUM_NOT_IMPLEMENTED. */
int32_t stratum_b200_debug_bpm_grid(float min_bpm, float max_bpm, float bpm_resolution, float* out, int32_t cap);

/* Per-stage device time (ms) accumulated since the last reset; names newline separated. */
int32_t stratum_b200_stage_times(char* names, size_t cap, double* ms, int32_t max_stages);
void stratum_b200_stage_times_reset(void);
void stratum_b200_stage_timing_enable(int32_t on);

/* Device time (CUDA events on the library's own stream, first launch to last copy, summed over the
 * waves) of the most recent stratum_b200_analyze_batch_device call in this process. */
double stratum_b200_last_call_device_ms(void);

/* Number of waves (arena-sized sub-batches = launches of every stage kernel) the most recent batch call was cut into. */
uint32_t stratum_b200_last_call_waves(void);

/* Cumulative host->device / device->host bytes copied by the library in this process. */
void stratum_b200_transfer_bytes(uint64_t* h2d, uint64_t* d2h);

#ifdef __cplusplus
}
#endif
#endif /* STRATUM_B200_H */
