"""float64 reference of album loudness (include/stratum_b200.h: stratum_b200_loudness_albums_pcm), written from the definitions on
top of loudness_ref.py: the members' momentary and short-term powers concatenated in track order, then the per-track gates, maxima
and percentile rule on the pooled lists."""
from __future__ import annotations

import math

import numpy as np
from scipy.signal import lfilter

import loudness_ref as R
import stratum_dsp_b200 as S


def blocks(t: S.PcmTrack):
    """(decoded f64 samples (frames, C), momentary powers m[0..J), short-term powers q[0..K)) of one track, as loudness_ref.measure
    forms them."""
    sr = t.sample_rate
    x = R.decode(t).astype(np.float64)
    frames, C = x.shape
    Sb = (sr + 5) // 10
    (b1, a1), (b2, a2) = R.kweight(sr)
    y = lfilter(b2, a2, lfilter(b1, a1, x, axis=0), axis=0)
    nfull = frames // Sb
    e = (y[: nfull * Sb] ** 2).reshape(nfull, Sb, C).sum(axis=1)
    z = e @ R.weights(C)
    J, K = max(0, nfull - 3), max(0, nfull - 29)
    mom = np.array([z[j:j + 4].sum() for j in range(J)]) / (4 * Sb)
    sht = np.array([z[k:k + 30].sum() for k in range(K)]) / (30 * Sb)
    return x, mom, sht


def gates(mom: np.ndarray, sht: np.ndarray) -> dict:
    """Integrated loudness, maxima and loudness range of a momentary and a short-term list."""
    lufs = R._lufs
    J, K = mom.size, sht.size
    lm, ls = lufs(mom), lufs(sht)
    integ = -math.inf
    g = mom[lm > -70.0]
    if g.size:
        rel = lufs(g.mean()) - 10.0
        g2 = mom[(lm > -70.0) & (lm > rel)]
        if g2.size:
            integ = float(lufs(g2.mean()))
    lra = 0.0
    g = sht[ls > -70.0]
    if g.size:
        rel = lufs(g.mean()) - 20.0
        v = np.sort(ls[(ls > -70.0) & (ls > rel)])
        n = v.size
        if n >= 2:
            lra = float(v[int(math.floor((n - 1) * 0.95 + 0.5))] - v[int(math.floor((n - 1) * 0.10 + 0.5))])
    return dict(integrated_lufs=integ, momentary_max_lufs=float(lm.max()) if J else -math.inf,
                short_term_max_lufs=float(ls.max()) if K else -math.inf, loudness_range_lu=lra, n_momentary=J, n_short_term=K)


def measure_album(tracks, with_true_peak: bool = True) -> dict:
    """The album rule over the tracks in the given order: gates, maxima and range of the concatenated lists, peaks the maxima over
    the tracks, frames their sum."""
    moms, shts, sp, tp, frames = [], [], 0.0, 0.0, 0
    for t in tracks:
        x, mom, sht = blocks(t)
        moms.append(mom)
        shts.append(sht)
        frames += x.shape[0]
        s = float(np.max(np.abs(x))) if x.shape[0] else 0.0
        sp = max(sp, s)
        if with_true_peak:
            tp = max(tp, s, R.true_peak(x, R.oversampling(t.sample_rate)))
    out = gates(np.concatenate(moms), np.concatenate(shts))
    out["sample_peak"] = sp
    out["frames"] = frames
    if with_true_peak:
        out["true_peak"] = tp
    return out
