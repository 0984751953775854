"""float64 reference of the loudness series (include/stratum_b200.h: stratum_b200_loudness_series_pcm), written from the definitions:
the momentary / short-term powers of loudness_layout_ref.blocks, and per-segment sample and true peaks from np.convolve."""
from __future__ import annotations

import numpy as np

import loudness_layout_ref as RL
import loudness_ref as R
import stratum_dsp_b200 as S


def _lufs(p):
    with np.errstate(divide="ignore"):
        return -0.691 + 10.0 * np.log10(p)


def segment_peaks(x: np.ndarray, sr: int):
    """(sample peaks, true peaks) per segment of S = (sr + 5) // 10 frames over all channels of x (frames, C).  Frame n owns the
    oversampled outputs u[L n .. L n + L - 1] (u[L n] = x[n]: the taps interpolate)."""
    x = np.asarray(x, np.float64)
    frames, C = x.shape
    Sb = (sr + 5) // 10
    L = R.oversampling(sr)
    c = R.taps(L)
    a = np.abs(x).max(axis=1)
    t = a.copy()
    for ch in range(C):
        xz = np.zeros(L * frames)
        xz[::L] = x[:, ch]
        u = np.convolve(xz, c)[24:24 + L * frames]
        t = np.maximum(t, np.abs(u).reshape(frames, L).max(axis=1))
    starts = np.arange(0, frames, Sb)
    return np.maximum.reduceat(a, starts), np.maximum.reduceat(t, starts)


def series(t: S.PcmTrack, codes=None) -> dict:
    """The four series of track t under channel classes `codes` (None: the default map)."""
    x, mom, sht = RL.blocks(t, S.channel_map(0, t.channels) if codes is None else codes)
    sp, tp = segment_peaks(x, t.sample_rate)
    return dict(momentary_lufs=_lufs(mom), short_term_lufs=_lufs(sht), sample_peak=sp, true_peak=tp)
