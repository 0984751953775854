//! B200 backend for stratum-dsp's per-track analysis hot path.
//!
//! Same signatures as the reference (`stratum_dsp::analyze_audio`, `src/lib.rs:86-90`;
//! `compute_confidence`, `src/analysis/confidence.rs:121`) plus the batch surface of
//! `examples/analyze_batch.rs:260-326` as one call.  All arithmetic runs in hand-written CUDA
//! kernels behind `libstratum_b200.so`; there is no CPU fallback — without a CUDA device every call
//! returns `AnalysisError::ProcessingError`.
//!
//! ```no_run
//! use stratum_dsp::AnalysisConfig;
//! let samples: Vec<f32> = vec![0.0; 44_100 * 30];
//! let r = stratum_dsp_b200::analyze_audio(&samples, 44_100, AnalysisConfig::default())?;
//! let c = stratum_dsp_b200::compute_confidence(&r);
//! println!("{:.2} BPM, key {}, overall {:.2}", r.bpm, r.key.name(), c.overall_confidence);
//! # Ok::<(), stratum_dsp::AnalysisError>(())
//! ```
pub mod sys;

use std::os::raw::c_char;

use stratum_dsp::analysis::result::{AnalysisFlag, TempoCandidateDebug};
pub use stratum_dsp::{compute_confidence, AnalysisConfidence, AnalysisConfig, AnalysisError, AnalysisMetadata, AnalysisResult, BeatGrid, Key};

use sys::*;

fn check_abi() -> Result<(), AnalysisError> {
    let ok = unsafe {
        stratum_b200_sizeof(0) == std::mem::size_of::<StratumConfig>()
            && stratum_b200_sizeof(1) == std::mem::size_of::<StratumResult>()
            && stratum_b200_sizeof(2) == std::mem::size_of::<StratumConfidence>()
    };
    if ok {
        Ok(())
    } else {
        Err(AnalysisError::ProcessingError("libstratum_b200.so does not match this binding (struct sizes differ)".to_string()))
    }
}

fn c_string(buf: &[c_char]) -> String {
    let bytes: Vec<u8> = buf.iter().take_while(|&&b| b != 0).map(|&b| b as u8).collect();
    String::from_utf8_lossy(&bytes).into_owned()
}

fn last_error() -> String {
    let mut buf = [0 as c_char; 1024];
    unsafe { stratum_b200_last_error(buf.as_mut_ptr(), buf.len()) };
    c_string(&buf)
}

/// StratumStatus (1..5) to the `AnalysisError` variant of `src/error.rs:7-22`.
fn to_error(code: i32, msg: String) -> AnalysisError {
    match code {
        1 => AnalysisError::InvalidInput(msg),
        2 => AnalysisError::DecodingError(msg),
        4 => AnalysisError::NotImplemented(msg),
        5 => AnalysisError::NumericalError(msg),
        _ => AnalysisError::ProcessingError(msg),
    }
}

unsafe fn vec_of<T: Copy>(p: *const T, n: u32) -> Vec<T> {
    if p.is_null() || n == 0 {
        Vec::new()
    } else {
        std::slice::from_raw_parts(p, n as usize).to_vec()
    }
}

fn opt_bool(v: i32) -> Option<bool> {
    if v < 0 {
        None
    } else {
        Some(v != 0)
    }
}

/// One `StratumResult` to the reference's `AnalysisResult` (built like `src/lib.rs:1592-1619`).
fn from_c(r: &StratumResult, _cfg: &AnalysisConfig) -> AnalysisResult {
    let mut wbuf = [0 as c_char; 2048];
    unsafe { stratum_b200_warning_strings(r, wbuf.as_mut_ptr(), wbuf.len()) };
    // the exact strings of lib.rs:1567-1589 — compute_confidence matches on them (confidence.rs:231-297)
    let confidence_warnings: Vec<String> = c_string(&wbuf).lines().filter(|l| !l.is_empty()).map(|l| l.to_string()).collect();
    let mut flags = Vec::new();
    if r.flags & 1 != 0 {
        flags.push(AnalysisFlag::MultimodalBpm);
    }
    if r.flags & 2 != 0 {
        flags.push(AnalysisFlag::WeakTonality);
    }
    if r.flags & 4 != 0 {
        flags.push(AnalysisFlag::TempoVariation);
    }
    if r.flags & 8 != 0 {
        flags.push(AnalysisFlag::OnsetDetectionAmbiguous);
    }
    let tempogram_candidates = if r.n_tempogram_candidates < 0 {
        None
    } else {
        Some(
            unsafe { vec_of(r.tempogram_candidates as *const StratumTempoCandidate, r.n_tempogram_candidates as u32) }
                .iter()
                .map(|c| TempoCandidateDebug { bpm: c.bpm, score: c.score, fft_norm: c.fft_norm, autocorr_norm: c.autocorr_norm, selected: c.selected != 0 })
                .collect(),
        )
    };
    // the same three strings for every track, whatever the configuration (lib.rs:1604-1608)
    let methods_used = vec!["energy_flux".to_string(), "chroma_extraction".to_string(), "key_detection".to_string()];
    AnalysisResult {
        bpm: r.bpm,
        bpm_confidence: r.bpm_confidence,
        key: if r.key_is_minor != 0 { Key::Minor(r.key_index) } else { Key::Major(r.key_index) },
        key_confidence: r.key_confidence,
        key_clarity: r.key_clarity,
        beat_grid: BeatGrid {
            downbeats: unsafe { vec_of(r.downbeats as *const f32, r.n_downbeats) },
            beats: unsafe { vec_of(r.beats as *const f32, r.n_beats) },
            bars: unsafe { vec_of(r.bars as *const f32, r.n_bars) },
        },
        grid_stability: r.grid_stability,
        metadata: AnalysisMetadata {
            duration_seconds: r.duration_seconds,
            sample_rate: r.sample_rate,
            processing_time_ms: r.processing_time_ms,
            algorithm_version: "0.1.0-alpha".to_string(),
            onset_method_consensus: r.onset_method_consensus,
            methods_used,
            flags,
            confidence_warnings,
            tempogram_candidates,
            tempogram_multi_res_triggered: opt_bool(r.tempogram_multi_res_triggered),
            tempogram_multi_res_used: opt_bool(r.tempogram_multi_res_used),
            tempogram_percussive_triggered: opt_bool(r.tempogram_percussive_triggered),
            tempogram_percussive_used: opt_bool(r.tempogram_percussive_used),
        },
    }
}

/// `stratum_dsp::analyze_audio` (`src/lib.rs:86-90`) on the B200 path.
pub fn analyze_audio(samples: &[f32], sample_rate: u32, config: AnalysisConfig) -> Result<AnalysisResult, AnalysisError> {
    check_abi()?;
    let cfg = config_to_c(&config)?;
    let mut r: StratumResult = unsafe { std::mem::zeroed() };
    let st = unsafe { stratum_b200_analyze_audio(samples.as_ptr(), samples.len() as u64, sample_rate, &cfg, &mut r) };
    let out = if st == 0 {
        Ok(from_c(&r, &config))
    } else {
        let msg = c_string(&r.error);
        Err(to_error(st, if msg.is_empty() { last_error() } else { msg }))
    };
    unsafe { stratum_b200_result_free(&mut r, 1) };
    out
}

/// The batch surface of `examples/analyze_batch.rs:260-326` (`paths.par_iter().map(analyze_audio)`) as one call:
/// tracks are sharded across `devices` (empty = the current device), a failed track yields its own `Err` and never
/// aborts the batch (`ItemOut.ok` / `ItemOut.error`).  The outer `Err` is returned only when nothing could run.
pub fn analyze_batch(tracks: &[&[f32]], sample_rates: &[u32], config: AnalysisConfig, devices: &[i32]) -> Result<Vec<Result<AnalysisResult, AnalysisError>>, AnalysisError> {
    check_abi()?;
    if tracks.len() != sample_rates.len() {
        return Err(AnalysisError::InvalidInput("tracks and sample_rates differ in length".to_string()));
    }
    let cfg = config_to_c(&config)?;
    let n = tracks.len();
    let mut offsets = Vec::with_capacity(n + 1);
    offsets.push(0u64);
    for t in tracks {
        offsets.push(offsets.last().unwrap() + t.len() as u64);
    }
    // one contiguous host buffer (a caller that decodes straight into pinned memory can use `sys` directly)
    let mut flat: Vec<f32> = Vec::with_capacity(*offsets.last().unwrap() as usize);
    for t in tracks {
        flat.extend_from_slice(t);
    }
    let mut res: Vec<StratumResult> = vec![unsafe { std::mem::zeroed() }; n];
    let st = unsafe {
        stratum_b200_analyze_batch(flat.as_ptr(), offsets.as_ptr(), sample_rates.as_ptr(), n as u32, &cfg,
                                   if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() }, devices.len() as u32, res.as_mut_ptr())
    };
    if st != 0 {
        let e = to_error(st, last_error());
        unsafe { stratum_b200_result_free(res.as_mut_ptr(), n as u32) }; // waves that completed before the error own heap arrays
        return Err(e);
    }
    let out = res.iter().map(|r| if r.status == 0 { Ok(from_c(r, &config)) } else { Err(to_error(r.status, c_string(&r.error))) }).collect();
    unsafe { stratum_b200_result_free(res.as_mut_ptr(), n as u32) };
    Ok(out)
}

/// One track of undecoded interleaved PCM for `loudness_batch_pcm`: `data` holds whole sample frames, little-endian, 24-bit
/// samples packed in 3 bytes; `format` is a `STRATUM_PCM_*` value (1 = u8 ... 6 = f64).
pub struct PcmTrack<'a> {
    pub data: &'a [u8],
    pub format: u32,
    pub channels: u32,
    pub sample_rate: u32,
}

/// ITU-R BS.1770-4 / EBU R128 loudness of one track (`StratumLoudness` in `include/stratum_b200.h`): LUFS, LU and linear peaks;
/// undefined loudness values are `f64::NEG_INFINITY`.
#[derive(Clone, Copy, Debug, PartialEq)]
pub struct Loudness {
    pub integrated_lufs: f64,
    pub momentary_max_lufs: f64,
    pub short_term_max_lufs: f64,
    pub loudness_range_lu: f64,
    pub sample_peak: f64,
    pub true_peak: f64,
    pub n_momentary: u32,
    pub n_short_term: u32,
}

/// Loudness of a batch of PCM tracks, measured on the device and sharded over `devices` (empty: the current device).  The outer
/// error rejects the whole call (no device, malformed input); a track that fails on its own carries its error in its slot.
pub fn loudness_batch_pcm(tracks: &[PcmTrack], devices: &[i32]) -> Result<Vec<Result<Loudness, AnalysisError>>, AnalysisError> {
    loudness_albums_pcm(tracks, &vec![None; tracks.len()], devices).map(|(per_track, _)| per_track)
}

/// Per-track loudness plus the loudness of albums (ReplayGain / R128 album values): `albums[i]` is the album of track i (`None`: no
/// album), ids from 0; there are max id + 1 albums.  Each album is measured over the pooled 400 ms blocks and 3 s windows of its
/// members, so its integrated loudness and range are not functions of the track values.  An album with a failed member, or an id no
/// track names, carries its error in its slot.
pub fn loudness_albums_pcm(tracks: &[PcmTrack], albums: &[Option<u32>], devices: &[i32])
    -> Result<(Vec<Result<Loudness, AnalysisError>>, Vec<Result<Loudness, AnalysisError>>), AnalysisError> {
    loudness_mapped_pcm(tracks, albums, None, false, devices).map(|(per_track, per_album, _)| (per_track, per_album))
}

/// Per-channel results of `loudness_mapped_pcm`: for each track, one `Loudness` per channel, each channel measured alone at weight
/// 1.0 (empty without `per_channel`).
pub type PerChannel = Vec<Vec<Result<Loudness, AnalysisError>>>;

/// The BS.1770-4 channel classes (`STRATUM_CH_*`) of a track of `channels` channels from its WAVE_FORMAT_EXTENSIBLE channel mask
/// (0: the default map of the channel count); `dual_mono` weighs a one-channel track as a mono signal on two loudspeakers.
pub fn channel_map(wave_mask: u32, channels: u32, dual_mono: bool) -> Result<Vec<u8>, AnalysisError> {
    let mut map = vec![0u8; channels.max(1) as usize];
    let st = unsafe { stratum_b200_loudness_channel_map(wave_mask, channels, dual_mono as i32, map.as_mut_ptr()) };
    if st != 0 {
        return Err(to_error(st, last_error()));
    }
    Ok(map)
}

/// `loudness_albums_pcm` with channel maps and per-channel results: `channel_maps[i]` holds track i's channel classes (`None`: its
/// default map; `channel_maps = None`: the default map for every track); with `per_channel` the third list holds each track's
/// channels measured alone.  Albums pool their members' mapped powers.
pub fn loudness_mapped_pcm(tracks: &[PcmTrack], albums: &[Option<u32>], channel_maps: Option<&[Option<Vec<u8>>]>, per_channel: bool, devices: &[i32])
    -> Result<(Vec<Result<Loudness, AnalysisError>>, Vec<Result<Loudness, AnalysisError>>, PerChannel), AnalysisError> {
    check_loudness_abi()?;
    let (ids, n_albums) = album_ids(albums, tracks.len())?;
    let n = tracks.len();
    let (flat, offsets, srs, chans, fmts) = pcm_tables(tracks);
    let map = flat_channel_map(channel_maps, &chans)?;
    let mut res: Vec<StratumLoudness> = vec![unsafe { std::mem::zeroed() }; n];
    let mut alb: Vec<StratumLoudness> = vec![unsafe { std::mem::zeroed() }; n_albums];
    let mut chout: Vec<StratumLoudness> = vec![unsafe { std::mem::zeroed() }; if per_channel { chans.iter().map(|&c| c as usize).sum() } else { 0 }];
    let st = unsafe {
        stratum_b200_loudness_mapped_pcm(flat.as_ptr(), offsets.as_ptr(), srs.as_ptr(), chans.as_ptr(), fmts.as_ptr(), n as u32, ids.as_ptr(),
                                         n_albums as u32, map.as_ref().map_or(std::ptr::null(), |m| m.as_ptr()),
                                         if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() }, devices.len() as u32,
                                         res.as_mut_ptr(), alb.as_mut_ptr(), if per_channel { chout.as_mut_ptr() } else { std::ptr::null_mut() })
    };
    if st != 0 {
        return Err(to_error(st, last_error()));
    }
    Ok((res.iter().map(loudness_from_c).collect(), alb.iter().map(loudness_from_c).collect(), split_channels(&chout, &chans, per_channel)))
}

/// The loudness series of one track (`stratum_b200_loudness_series_pcm` in `include/stratum_b200.h`) at a step of `step_seconds` =
/// S / sr, S = (sr + 5) / 10 frames: `momentary_lufs[j]` is the 400 ms block [jS, jS + 4S) (a meter shows it at (j + 4) S / sr),
/// `short_term_lufs[k]` the 3 s window [kS, kS + 30S), `sample_peak[s]` / `true_peak[s]` the linear peaks over all channels of the
/// frames [sS, (s + 1) S).  The largest entries equal the track's maxima and peaks.
#[derive(Clone, Debug, PartialEq)]
pub struct LoudnessSeries {
    pub momentary_lufs: Vec<f64>,
    pub short_term_lufs: Vec<f64>,
    pub sample_peak: Vec<f64>,
    pub true_peak: Vec<f64>,
    pub step_seconds: f64,
}

/// `loudness_mapped_pcm` without albums or per-channel results, plus each measured track's loudness series.
#[allow(clippy::type_complexity)]
pub fn loudness_series_pcm(tracks: &[PcmTrack], channel_maps: Option<&[Option<Vec<u8>>]>, devices: &[i32])
    -> Result<Vec<Result<(Loudness, LoudnessSeries), AnalysisError>>, AnalysisError> {
    check_loudness_abi()?;
    let n = tracks.len();
    let (flat, offsets, srs, chans, fmts) = pcm_tables(tracks);
    let map = flat_channel_map(channel_maps, &chans)?;
    let mut lens = Vec::with_capacity(n);
    for (i, t) in tracks.iter().enumerate() {
        let sample_bytes: u64 = match t.format { 1 => 1, 2 => 2, 3 => 3, 4 | 5 => 4, 6 => 8, _ => 0 };  // an unknown format is rejected by the call
        let bpf = sample_bytes * t.channels.max(1) as u64;
        let frames = if bpf > 0 { (offsets[i + 1] - offsets[i]) / bpf } else { 0 };
        let (mut m, mut q, mut p) = (0u32, 0u32, 0u32);
        unsafe { stratum_b200_loudness_series_lengths(t.sample_rate, frames, &mut m, &mut q, &mut p) };
        lens.push((m as usize, q as usize, p as usize));
    }
    let mut mom = vec![0.0f64; lens.iter().map(|l| l.0).sum()];
    let mut sht = vec![0.0f64; lens.iter().map(|l| l.1).sum()];
    let mut spk = vec![0.0f64; lens.iter().map(|l| l.2).sum()];
    let mut tpk = vec![0.0f64; spk.len()];
    let mut res: Vec<StratumLoudness> = vec![unsafe { std::mem::zeroed() }; n];
    let st = unsafe {
        stratum_b200_loudness_series_pcm(flat.as_ptr(), offsets.as_ptr(), srs.as_ptr(), chans.as_ptr(), fmts.as_ptr(), n as u32, std::ptr::null(), 0,
                                         map.as_ref().map_or(std::ptr::null(), |m| m.as_ptr()),
                                         if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() }, devices.len() as u32,
                                         res.as_mut_ptr(), std::ptr::null_mut(), std::ptr::null_mut(), mom.as_mut_ptr(), sht.as_mut_ptr(), spk.as_mut_ptr(),
                                         tpk.as_mut_ptr())
    };
    if st != 0 {
        return Err(to_error(st, last_error()));
    }
    let (mut a, mut b, mut c) = (0usize, 0usize, 0usize);
    Ok(res.iter().zip(lens).map(|(r, (m, q, p))| {
        let series = LoudnessSeries {
            momentary_lufs: mom[a..a + m].to_vec(),
            short_term_lufs: sht[b..b + q].to_vec(),
            sample_peak: spk[c..c + p].to_vec(),
            true_peak: tpk[c..c + p].to_vec(),
            step_seconds: if r.sample_rate > 0 { ((r.sample_rate + 5) / 10) as f64 / r.sample_rate as f64 } else { 0.0 },
        };
        a += m;
        b += q;
        c += p;
        loudness_from_c(r).map(|l| (l, series))
    }).collect())
}

/// Analysis (as `analyze_batch` gives it) and loudness (as `loudness_albums_pcm` gives it) of the same PCM tracks from one upload of
/// each byte.  `albums`: as in `loudness_albums_pcm`, or `None` for no albums (the album list is then empty).  A track's analysis
/// and its loudness fail or succeed independently.
pub fn analyze_loudness_pcm(tracks: &[PcmTrack], albums: Option<&[Option<u32>]>, config: AnalysisConfig, devices: &[i32])
    -> Result<(Vec<Result<AnalysisResult, AnalysisError>>, Vec<Result<Loudness, AnalysisError>>, Vec<Result<Loudness, AnalysisError>>), AnalysisError> {
    analyze_loudness_mapped_pcm(tracks, albums, None, false, config, devices).map(|(results, per_track, per_album, _)| (results, per_track, per_album))
}

/// `analyze_loudness_pcm` with `channel_maps` and `per_channel` as in `loudness_mapped_pcm`; the maps weigh the loudness only (the
/// analysis mixdown stays the equal-weight average).
#[allow(clippy::type_complexity)]
pub fn analyze_loudness_mapped_pcm(tracks: &[PcmTrack], albums: Option<&[Option<u32>]>, channel_maps: Option<&[Option<Vec<u8>>]>, per_channel: bool,
                                   config: AnalysisConfig, devices: &[i32])
    -> Result<(Vec<Result<AnalysisResult, AnalysisError>>, Vec<Result<Loudness, AnalysisError>>, Vec<Result<Loudness, AnalysisError>>, PerChannel),
              AnalysisError> {
    check_abi()?;
    check_loudness_abi()?;
    let cfg = config_to_c(&config)?;
    let n = tracks.len();
    let (ids, n_albums) = match albums {
        Some(a) => album_ids(a, n)?,
        None => (Vec::new(), 0),
    };
    let (flat, offsets, srs, chans, fmts) = pcm_tables(tracks);
    let map = flat_channel_map(channel_maps, &chans)?;
    let mut res: Vec<StratumResult> = vec![unsafe { std::mem::zeroed() }; n];
    let mut loud: Vec<StratumLoudness> = vec![unsafe { std::mem::zeroed() }; n];
    let mut alb: Vec<StratumLoudness> = vec![unsafe { std::mem::zeroed() }; n_albums];
    let mut chout: Vec<StratumLoudness> = vec![unsafe { std::mem::zeroed() }; if per_channel { chans.iter().map(|&c| c as usize).sum() } else { 0 }];
    let st = unsafe {
        stratum_b200_analyze_loudness_mapped_pcm(flat.as_ptr(), offsets.as_ptr(), srs.as_ptr(), chans.as_ptr(), fmts.as_ptr(), n as u32, &cfg,
                                                 if albums.is_some() { ids.as_ptr() } else { std::ptr::null() }, n_albums as u32,
                                                 map.as_ref().map_or(std::ptr::null(), |m| m.as_ptr()),
                                                 if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() }, devices.len() as u32,
                                                 res.as_mut_ptr(), loud.as_mut_ptr(), alb.as_mut_ptr(),
                                                 if per_channel { chout.as_mut_ptr() } else { std::ptr::null_mut() })
    };
    if st != 0 {
        let e = to_error(st, last_error());
        unsafe { stratum_b200_result_free(res.as_mut_ptr(), n as u32) }; // waves that completed before the error own heap arrays
        return Err(e);
    }
    let out = res.iter().map(|r| if r.status == 0 { Ok(from_c(r, &config)) } else { Err(to_error(r.status, c_string(&r.error))) }).collect();
    unsafe { stratum_b200_result_free(res.as_mut_ptr(), n as u32) };
    Ok((out, loud.iter().map(loudness_from_c).collect(), alb.iter().map(loudness_from_c).collect(), split_channels(&chout, &chans, per_channel)))
}

/// The maps of the tracks in one buffer for the C call (`None` entries filled with the default map), or `None` for no map.
fn flat_channel_map(channel_maps: Option<&[Option<Vec<u8>>]>, chans: &[u32]) -> Result<Option<Vec<u8>>, AnalysisError> {
    let Some(maps) = channel_maps else { return Ok(None) };
    if maps.len() != chans.len() {
        return Err(AnalysisError::InvalidInput("one channel map (or None) per track".to_string()));
    }
    let mut flat = Vec::new();
    for (i, (m, &c)) in maps.iter().zip(chans).enumerate() {
        let m = match m {
            Some(m) => m.clone(),
            None => channel_map(0, c, false)?,
        };
        if m.len() != c as usize {
            return Err(AnalysisError::InvalidInput(format!("track {i}: {} channel classes for {c} channels", m.len())));
        }
        flat.extend_from_slice(&m);
    }
    Ok(Some(flat))
}

fn split_channels(chout: &[StratumLoudness], chans: &[u32], per_channel: bool) -> PerChannel {
    if !per_channel {
        return chans.iter().map(|_| Vec::new()).collect();
    }
    let mut at = 0usize;
    chans.iter().map(|&c| {
        let v = chout[at..at + c as usize].iter().map(loudness_from_c).collect();
        at += c as usize;
        v
    }).collect()
}

fn check_loudness_abi() -> Result<(), AnalysisError> {
    if unsafe { stratum_b200_sizeof(3) } != std::mem::size_of::<StratumLoudness>() {
        return Err(AnalysisError::ProcessingError("libstratum_b200.so does not match this binding (struct sizes differ)".to_string()));
    }
    Ok(())
}

/// Album ids for the C call (`None` -> `STRATUM_NO_ALBUM`) and the album count, max id + 1.
fn album_ids(albums: &[Option<u32>], n_tracks: usize) -> Result<(Vec<u32>, usize), AnalysisError> {
    if albums.len() != n_tracks {
        return Err(AnalysisError::InvalidInput("one album id (or None) per track".to_string()));
    }
    let ids: Vec<u32> = albums.iter().map(|a| a.unwrap_or(STRATUM_NO_ALBUM)).collect();
    let n_albums = albums.iter().flatten().map(|a| *a as u64 + 1).max().unwrap_or(0);
    if n_albums > u32::MAX as u64 {
        return Err(AnalysisError::InvalidInput("album id STRATUM_NO_ALBUM is reserved for None".to_string()));
    }
    Ok((ids, n_albums as usize))
}

/// The tracks' bytes in one buffer, their byte offsets, sample rates, channel counts and formats.
fn pcm_tables(tracks: &[PcmTrack]) -> (Vec<u8>, Vec<u64>, Vec<u32>, Vec<u32>, Vec<u32>) {
    let mut offsets = vec![0u64];
    let mut flat: Vec<u8> = Vec::new();
    for t in tracks {
        flat.extend_from_slice(t.data);
        offsets.push(flat.len() as u64);
    }
    let srs: Vec<u32> = tracks.iter().map(|t| t.sample_rate).collect();
    let chans: Vec<u32> = tracks.iter().map(|t| t.channels).collect();
    let fmts: Vec<u32> = tracks.iter().map(|t| t.format).collect();
    (flat, offsets, srs, chans, fmts)
}

fn loudness_from_c(r: &StratumLoudness) -> Result<Loudness, AnalysisError> {
    if r.status != 0 {
        return Err(to_error(r.status, c_string(&r.error)));
    }
    Ok(Loudness {
        integrated_lufs: r.integrated_lufs,
        momentary_max_lufs: r.momentary_max_lufs,
        short_term_max_lufs: r.short_term_max_lufs,
        loudness_range_lu: r.loudness_range_lu,
        sample_peak: r.sample_peak,
        true_peak: r.true_peak,
        n_momentary: r.n_momentary,
        n_short_term: r.n_short_term,
    })
}

/// Decoder-side batch entry: interleaved 16-bit PCM uploaded as is and converted on the device with the arithmetic of
/// `examples/analyze_batch.rs:96-113` (half the PCIe bytes of f32).
pub fn analyze_batch_pcm16(tracks: &[&[i16]], sample_rates: &[u32], channels: &[u32], config: AnalysisConfig, devices: &[i32]) -> Result<Vec<Result<AnalysisResult, AnalysisError>>, AnalysisError> {
    check_abi()?;
    if tracks.len() != sample_rates.len() || tracks.len() != channels.len() {
        return Err(AnalysisError::InvalidInput("tracks, sample_rates and channels differ in length".to_string()));
    }
    let cfg = config_to_c(&config)?;
    let n = tracks.len();
    let mut offsets = vec![0u64];
    for t in tracks {
        offsets.push(offsets.last().unwrap() + t.len() as u64);
    }
    let mut flat: Vec<i16> = Vec::with_capacity(*offsets.last().unwrap() as usize);
    for t in tracks {
        flat.extend_from_slice(t);
    }
    let mut res: Vec<StratumResult> = vec![unsafe { std::mem::zeroed() }; n];
    let st = unsafe {
        stratum_b200_analyze_batch_pcm16(flat.as_ptr(), offsets.as_ptr(), sample_rates.as_ptr(), channels.as_ptr(), n as u32, &cfg,
                                         if devices.is_empty() { std::ptr::null() } else { devices.as_ptr() }, devices.len() as u32, res.as_mut_ptr())
    };
    if st != 0 {
        let e = to_error(st, last_error());
        unsafe { stratum_b200_result_free(res.as_mut_ptr(), n as u32) }; // waves that completed before the error own heap arrays
        return Err(e);
    }
    let out = res.iter().map(|r| if r.status == 0 { Ok(from_c(r, &config)) } else { Err(to_error(r.status, c_string(&r.error))) }).collect();
    unsafe { stratum_b200_result_free(res.as_mut_ptr(), n as u32) };
    Ok(out)
}
