"""float64 reference of the loudness measurement with explicit channel weights (include/stratum_b200.h: StratumChannelClass), on top
of loudness_ref.py and loudness_album_ref.py: the same K-weighting, blocks, gates and peaks, with the power summed as
sum_c w_c * mean(y_c^2) for the weights of a channel map instead of the default map."""
from __future__ import annotations

import numpy as np
from scipy.signal import lfilter

import loudness_album_ref as RA
import loudness_ref as R
import stratum_dsp_b200 as S

CLASS_WEIGHT = {S.CH_UNUSED: 0.0, S.CH_FRONT: 1.0, S.CH_SURROUND: 1.41, S.CH_DUAL_MONO: 2.0}


def weights(codes) -> np.ndarray:
    return np.array([CLASS_WEIGHT[int(c)] for c in codes])


def blocks(t: S.PcmTrack, codes):
    """(decoded f64 samples, momentary powers, short-term powers) of one track weighted by the classes `codes`."""
    sr = t.sample_rate
    x = R.decode(t).astype(np.float64)
    frames, C = x.shape
    Sb = (sr + 5) // 10
    (b1, a1), (b2, a2) = R.kweight(sr)
    y = lfilter(b2, a2, lfilter(b1, a1, x, axis=0), axis=0)
    nfull = frames // Sb
    e = (y[: nfull * Sb] ** 2).reshape(nfull, Sb, C).sum(axis=1)
    z = e @ weights(codes)
    J, K = max(0, nfull - 3), max(0, nfull - 29)
    mom = np.array([z[j:j + 4].sum() for j in range(J)]) / (4 * Sb)
    sht = np.array([z[k:k + 30].sum() for k in range(K)]) / (30 * Sb)
    return x, mom, sht


def measure(t: S.PcmTrack, codes) -> dict:
    """loudness_ref.measure with the weights of `codes`; the peaks stay the maxima over every channel."""
    return measure_album([t], [codes])


def measure_album(tracks, maps) -> dict:
    """loudness_album_ref.measure_album with track i weighted by maps[i]."""
    moms, shts, sp, tp, frames = [], [], 0.0, 0.0, 0
    for t, codes in zip(tracks, maps):
        x, mom, sht = blocks(t, codes)
        moms.append(mom)
        shts.append(sht)
        frames += x.shape[0]
        s = float(np.max(np.abs(x))) if x.shape[0] else 0.0
        sp = max(sp, s)
        tp = max(tp, s, R.true_peak(x, R.oversampling(t.sample_rate)))
    out = RA.gates(np.concatenate(moms), np.concatenate(shts))
    out.update(sample_peak=sp, true_peak=tp, frames=frames)
    return out


def channel_track(t: S.PcmTrack, c: int) -> S.PcmTrack:
    """The one-channel track holding exactly channel c's bytes of t."""
    b = S._PCM_BYTES[t.fmt]
    d = np.ascontiguousarray(t.data.reshape(-1, t.channels, b)[:, c, :]).reshape(-1)
    return S.PcmTrack(d, t.fmt, 1, t.sample_rate)
