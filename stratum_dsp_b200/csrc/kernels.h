// Host-side launch interface of the kernel translation units.
#pragma once
#include "common.cuh"

namespace sb {

// Values of StratumConfig that kernels read (copied by value into launches).
struct DevCfg {
    float min_bpm, max_bpm, bpm_resolution;
    // BPM hypothesis grid, built on the host with the reference's f32 accumulation (engine.cu: bpm_grid)
    uint32_t n_bpm;               // autocorrelation tempogram: `bpm <= max_bpm` (tempogram_autocorr.rs:79-178)
    uint32_t n_comb;              // comb filterbank: `bpm <= max_bpm + 1e-10` (comb_filter.rs:96-215)
    uint32_t ac_stride;           // floats per variant of HopLayout::tgac: max(AC_CAP, n_bpm)
    const float* bpm_tab;         // max(n_bpm, n_comb) hypothesis BPMs on the device; set only on the fine-grid path (either count > AC_CAP)
    float silence_thr_linear;     // 10^(min_amplitude_db/20), silence.rs:141
    uint32_t silence_min_ms;      // 500, lib.rs:134
    float energy_thr_mul;         // 10^(-20/20), energy_flux.rs:160
    float target_peak;            // 10^(-1/20), normalization.rs:290
    float rms_target;             // 10^((target_lufs + 3 - headroom)/20), normalization.rs:345 via :532
    int32_t normalization, enable_normalization, enable_trim, enable_consensus;
    float onset_pct;
    uint32_t consensus_tol_ms;
    float cons_w[4];
    int32_t hpss_onsets, perc_fallback, emit_cands;
    uint32_t hpss_margin;
    uint32_t hop;                 // hop_size of the base path (config.rs: 512)
    uint32_t frame, bins;         // frame_size of the tempo path (2048, 4096 or 8192: tempo_frame_supported) and its bin count frame/2 + 1
    int32_t bs;                   // slot of the base path: 0 (hop 512, shared with the multi-resolution pass) or SLOT_BASE_ALT
    uint32_t sf_k, mel_k;
    float nov_ws, nov_we, nov_wh;
    uint32_t nov_lmw, nov_smw;
    int32_t band_fusion, mel_enabled, seed_only;
    float w_full, w_low, w_mid, w_high, w_mel;
    float support_thr, consensus_bonus;
    uint32_t base_top_n, mr_top_k, mr_aux_k;
    float mr_w512, mr_w256, mr_w1024, mr_dt, mr_margin;
    int32_t mr_human_prior, mr_enabled;
    int32_t force_legacy, legacy_guardrails, bpm_fusion;
    float lg_pmin, lg_pmax, lg_smin, lg_smax, lg_mp, lg_ms, lg_me;
    // key
    uint32_t key_frame, key_hop, key_bins;  // key STFT geometry (lib.rs:984-995): override values or frame_size / hop_size; bins = frame/2 + 1
    uint32_t key_stride;          // floats per key-spectrogram row: key_bins, or (key_compact) rounded up to a 32-byte sector so that row loads are sector-aligned
    uint32_t key_margin;
    float key_mask_power;
    int32_t key_mask, key_weighting, key_voting;
    int32_t key_smooth_only;      // harmonic mask off, time smoothing on: the key spectrogram is replaced by its +-margin mean (lib.rs:1043-1060)
    int32_t key_hpcp;             // 0 = plain chroma folding (extractor.rs:393-487)
    int32_t key_compact;          // the mask writes the HPCP band + per-CTA frame-energy shares instead of rewriting the spectrogram (k_key.cu)
    float chroma_sharpen;         // > 1: sharpen_chroma (chroma/normalization.rs:41-65)
    float key_min_tonal, key_tonal_pow, key_energy_pow;
    uint32_t key_seg_len, key_seg_hop;
    float key_seg_min_clarity;
    uint32_t hpcp_peaks, hpcp_harm;
    float hpcp_decay, hpcp_pow, hpcp_sigma;
    // optional key scoring variants (SURVEY §8a a39)
    int32_t key_mode;             // KEY_ROWS_* (key_rows.cuh): segment voting / multi-scale / ensemble
    int32_t key_template_set;     // 0 = Krumhansl-Kessler, 1 = Temperley (key/templates.rs:16-22)
    int32_t key_edge_trim;
    float key_edge_frac;
    int32_t key_heur;             // detect_key_weighted_mode_heuristic replaces detect_key_weighted (lib.rs:1353-1372)
    float key_third_margin, key_flip_ratio;  // flip ratio is 0 unless enable_key_mode_heuristic (lib.rs:1361-1365)
    int32_t key_minor_bonus;
    float key_minor_bonus_w;
    float key_ens_kk, key_ens_tp;
    uint32_t ms_n, ms_len[8], ms_hop, ms_nw;
    float ms_w[8], ms_min_clarity;
    // optional chroma-side variants
    int32_t key_tuning;           // estimate_tuning_offset_semitones_from_spectrogram (extractor.rs:66-170)
    float tune_max_abs, tune_thr;
    uint32_t tune_step;
    int32_t key_whiten;           // enable_whitening && smooth_bins >= 3 (extractor.rs:562)
    uint32_t whiten_half;         // (max(smooth_bins, 3) | 1) / 2
    int32_t key_bass_blend;
    float bass_weight;
    int32_t key_log_freq, key_beat_sync, key_soft_mapping;
    int32_t key_hpss;             // harmonic_spectrogram_hpss_median_mask (extractor.rs:1369-1501)
    uint32_t khpss_step, khpss_tm, khpss_fm;
    float khpss_power;
};

// Frame sizes of the tempo path (silence detector, energy flux, STFT and its feature kernels).  2048 is the default; 4096 and 8192
// buy bass resolution.  Kernels that depend on the frame size are instantiated for exactly these three and dispatched by with_frame.
__host__ __device__ inline bool tempo_frame_supported(uint32_t frame) { return frame == 2048 || frame == 4096 || frame == 8192; }

// Frames of `frame` samples at `hop` in n samples (compute_stft, extractor.rs:301-359): the one frame-count rule of host and device.
__host__ __device__ inline uint32_t frames_of(uint64_t n, uint32_t frame, uint32_t hop) { return n >= frame ? (uint32_t)((n - frame) / hop + 1) : 0; }

template <int N>
struct FrameC {
    static constexpr int F = N, B = N / 2 + 1;
};
// Calls fn(FrameC<F>{}) with the configuration's frame size as a compile-time constant.
template <class Fn>
inline void with_frame(uint32_t frame, Fn&& fn) {
    if (frame == 8192) fn(FrameC<8192>{});
    else if (frame == 4096) fn(FrameC<4096>{});
    else fn(FrameC<2048>{});
}

// Grids of more than AC_CAP hypotheses take the fine-grid kernels (distinct-lag tempogram, table lookups, comb filterbank across CTAs).
__host__ __device__ inline bool fine_bpm_grid(const DevCfg& d) { return d.bpm_tab != nullptr; }

// Per-sample-rate tables (band edges, mel filterbank) — novelty.rs:72-190, tempogram.rs:364-372.
struct SrTables {
    uint32_t sr;
    uint32_t b0, b_low, b_mid, b_hi;  // band edges in bins of the 2048-point STFT
    uint32_t variant_mask;            // bit v set when variant v (full, low, mid, high, mel) is active
    uint32_t n_mels;
    const int32_t* mel_off;           // [n_mels + 1] entry ranges per mel band
    const int32_t* mel_bin;           // flat entries in ascending-bin order per band (centre bin twice: rising and falling slope)
    const float* mel_w;
    const int32_t* mel_chunks;        // fold schedule of par_feat_kernel (engine.cu: sr_slot): 64 chunks (first, end, position) + 41 band starts
    uint32_t key_bin_lo, key_bin_hi;  // HPCP peak search range in the key STFT (extractor.rs:584-591)
    uint32_t fold_lo, fold_hi;        // chroma-folding bin range (extractor.rs:407-417); lo > hi = empty
    const int32_t* fold_off;          // [13] entry ranges per pitch class
    const int32_t* fold_bin;          // entries in ascending-bin order per pitch class
    const float* fold_w;              // Gaussian (soft) or unit (hard) weights
    // optional key-path variants (SURVEY §8a a39), all in key-STFT bins
    uint32_t bass_bin_lo, bass_bin_hi;  // bass-band HPCP peak range (extractor.rs:1206-1220); lo > hi = empty
    float bass_fmin, bass_fmax;         // band edges after the clamps of extractor.rs:551-556
    uint32_t tune_bin_lo, tune_bin_hi;  // tuning estimator band, 80..2000 Hz (extractor.rs:100-121)
    uint32_t white_n;                   // whitened bins [0, white_n) a frame needs (peak tests read one bin past each band)
    uint32_t hpss_b0, hpss_band;        // median-HPSS band (extractor.rs:1408-1420); band = 0: spectrogram passes through
    uint32_t log_n;                     // semitone bins of the log-frequency spectrogram (extractor.rs:741-745)
    int32_t log_offset;                 // semitone index of bin 0 (lib.rs:1076-1079)
    const int32_t* log_off;             // [log_n + 1] entry ranges per semitone bin
    const int32_t* log_bin;             // linear bins in ascending order per semitone bin
    const float* log_w;                 // interpolation weights (extractor.rs:786-797)
    float kw_b0, kw_b1, kw_b2, kw_a1, kw_a2;  // K-weighting biquad (normalization.rs:127-155)
    uint32_t lufs_block;              // (sr * 0.4) as usize, normalization.rs:198
};

// Tables of the generic STFT (k_stft.cu: stft_any_kernel) for one frame size N = 2^m: Hann window, TW_{N/2} and the real-split table RW_N.
struct GenStft {
    const float* win;
    const float2* tw;
    const float2* rw;
    uint32_t n;
};

struct WaveCtx {
    cudaStream_t stream;
    const float* samples;  // device
    float* fa;             // float arena (work areas)
    float* oa;             // float output arena (beats, downbeats) — the only float region copied back
    int32_t* ia;           // int arena
    TrackDev* tracks;      // device
    const SrTables* srtab; // device array, tracks index it through sr_index
    const int32_t* sr_index;  // per track
    int n_tracks;
    Tables tab;
    DevCfg cfg;
    // maxima over the wave (grid sizing upper bounds)
    uint32_t max_F[N_SLOTS], max_Fk, max_Fsil;
    uint64_t max_n;
    uint32_t max_beat_cap;
    uint32_t max_seg_cap;
    uint32_t max_lg_fft;
    uint32_t max_lufs_nb;
    uint32_t max_key_peaks;  // HPCP peak slots a frame may need: (band bins + 1) / 2 over the wave's sample rates
    GenStft gen_key;         // key STFT frames other than 2048 / 8192 points (n = 0: unused)
    GenStft gen_tempo;       // tempo-path STFT tables at frame_size 4096 (n = 0: unused)
    uint32_t kband_stride_common;  // row stride of the compact key band when every live track of the wave has the same one, else 0
};

struct Launcher;  // counts launches + optional stage timing (engine.cu)
void count_launch(const char* stage);

// k_preprocess.cu
void launch_peak(const WaveCtx& c);
void launch_gain(const WaveCtx& c, const float* d_lufs_gain);
void launch_silence_trim(const WaveCtx& c);
// k_stft.cu
void launch_stft_hop(const WaveCtx& c, int hop_idx, const int32_t* d_list, int n_list);
void launch_stft_key(const WaveCtx& c);
void stft_upload_constants(const float2* ptw1024_host, const float2* ptw4096_host);  // per device, before the first STFT launch
void launch_stft_raw(cudaStream_t s, const float* d_samples, uint64_t n, uint32_t frame_size, uint32_t hop, float gain, const Tables& tab,
                     float* d_out, uint32_t frames, const GenStft* gen = nullptr);
// k_onset.cu
void launch_energy_onsets(const WaveCtx& c);
void launch_spec_features(const WaveCtx& c, int hop_idx, const int32_t* d_list, int n_list);
void launch_spectral_onsets_consensus(const WaveCtx& c);
// k_tempo.cu
void launch_tempogram(const WaveCtx& c, int hop_idx, const int32_t* d_list, int n_list);
void launch_escalation_gate(const WaveCtx& c);
void launch_escalation_compact(const WaveCtx& c, int32_t* d_list, int32_t* d_count, uint64_t slot_base, uint64_t slot_stride, uint32_t n_slots);
void launch_multires_fusion(const WaveCtx& c, const int32_t* d_list, int n_list);
void launch_final_bpm(const WaveCtx& c);
void launch_emit_candidates(const WaveCtx& c);
// k_legacy.cu
void launch_legacy_bpm(const WaveCtx& c);
// k_hpss.cu
void launch_hpss(const WaveCtx& c, const int32_t* d_list, int n_list);
void launch_hpss_onsets(const WaveCtx& c);
void launch_seq_features(const WaveCtx& c, int hop_idx, const int32_t* d_list, int n_list);
void launch_perc_accept(const WaveCtx& c, const int32_t* d_list, int n_list);
// k_beat.cu
void launch_beat_tracking(const WaveCtx& c);
// k_key.cu
void launch_key_mask(const WaveCtx& c);
void launch_key_hpcp(const WaveCtx& c);
void launch_key_vote(const WaveCtx& c);
void launch_key_variants_pre(const WaveCtx& c);  // k_keyvar.cu: median-HPSS mask, tuning estimate, whitening, per-track fold tables
void launch_key_chroma_variants(const WaveCtx& c);  // k_keyvar.cu: log-frequency chroma, beat-synchronous chroma
// k_loudness.cu: BS.1770-4 / EBU R128 loudness of interleaved PCM (stratum_b200_loudness_batch_pcm).
// One record per track of a launch, built on the host (engine.cu: loud_track).
struct LoudTrack {
    uint64_t byte_off;     // first byte of the track in the launch's PCM buffer
    uint64_t frames;
    uint64_t work;         // first work item (segment-major (segment, channel) pairs of the earlier tracks)
    uint64_t seg0;         // first entry in the per-segment work areas (segments of the earlier tracks)
    uint32_t C, fmt;       // channels, STRATUM_PCM_*
    uint32_t S, L;         // sub-block frames (sr + 5) / 10, true-peak oversampling factor
    uint32_t nseg, nfull;  // segments covering the track (0: the track failed and is skipped), whole sub-blocks floor(frames / S)
    uint32_t J, K;         // momentary blocks max(0, nfull - 3), short-term windows max(0, nfull - 29)
    double kw[10];         // K-weighting: stage 1 b0 b1 b2 a1 a2, stage 2 b0 b1 b2 a1 a2
    double M[16];          // A^S, row-major: maps the cascade state (z1, z2 of stage 1, z1, z2 of stage 2) across one silent sub-block
    float taps[49];        // true-peak interpolator
};
struct LoudOut {
    double integrated, momentary_max, short_term_max, loudness_range;
    uint32_t sample_peak_bits, true_peak_bits;  // non-negative floats, reduced by atomicMax on the bits
};
// libebur128's default channel map: 1 channel L; 4 channels L R Ls Rs; 5 channels L R C Ls Rs; otherwise L R C LFE Ls Rs and unused
// channels from 6 on.  L, R, C weigh 1, Ls and Rs 1.41, LFE and unused channels 0.
__host__ __device__ inline double loud_channel_weight(uint32_t C, uint32_t c) {
    if (C == 4) return c < 2 ? 1.0 : 1.41;
    if (C == 5) return c < 3 ? 1.0 : 1.41;
    if (c < 3) return 1.0;
    return (c == 4 || c == 5) ? 1.41 : 0.0;
}
void launch_loud_pass1(cudaStream_t s, const void* d_pcm, const LoudTrack* d_tr, uint32_t n_tracks, uint64_t n_work, double* d_st);
void launch_loud_scan(cudaStream_t s, const LoudTrack* d_tr, uint32_t n_tracks, uint32_t max_channels, double* d_st);
void launch_loud_pass2(cudaStream_t s, const void* d_pcm, const LoudTrack* d_tr, uint32_t n_tracks, uint64_t n_work, const double* d_st, double* d_en,
                       LoudOut* d_out);
// d_ws: 4 x n_seg doubles (sub-block, momentary and short-term powers, the compacted short-term powers of the loudness range)
void launch_loud_gate(cudaStream_t s, const LoudTrack* d_tr, uint32_t n_tracks, const double* d_en, double* d_ws, uint64_t n_seg, LoudOut* d_out);
// One record per album: its pooled momentary powers are mom[m0 .. m0 + J), its short-term powers sht[q0 .. q0 + K) (engine.cu:
// AlbumPools).  d_keep has the size of d_sht; only the loudness fields of d_out are written.
struct LoudAlbum {
    uint64_t m0, q0;
    uint32_t J, K;
};
void launch_loud_album_gate(cudaStream_t s, const LoudAlbum* d_al, uint32_t n_albums, const double* d_mom, const double* d_sht, double* d_keep,
                            LoudOut* d_out);
// k_synth.cu
void launch_pcm_to_mono(cudaStream_t s, const void* d_pcm, float* d_out, const uint64_t* d_byte_off, const uint64_t* d_out_off, const uint32_t* d_channels,
                        const uint32_t* d_formats, uint32_t n_tracks, uint64_t max_frames);
int check_divisions(cudaStream_t s, uint64_t n, uint32_t seed, unsigned long long* d_bad3);  // common.cuh divisions vs IEEE division (test instrumentation)
double measure_fp32_peak_tflops(cudaStream_t s, float* d_scratch);  // FMA microbenchmark (bench instrumentation)
void launch_synth(cudaStream_t s, float* d_out, uint32_t n_tracks, uint64_t n_samples, uint32_t sr, const float* d_params5);

}  // namespace sb
