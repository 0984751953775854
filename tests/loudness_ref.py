"""float64 reference of the BS.1770-4 / EBU R128 loudness measurement (include/stratum_b200.h: StratumLoudness), written from the
definitions: scipy.signal.lfilter over the whole track, numpy for blocks, gates and percentiles, np.convolve for the true peak.
PCM is converted to f32 exactly as the device converts it (csrc/pcm.cuh: pcm_sample), and PcmTrack encoders build test inputs."""
from __future__ import annotations

import math

import numpy as np
from scipy.signal import lfilter

import stratum_dsp_b200 as S


# ---- PCM ---------------------------------------------------------------------------------------------------------------
def encode(x: np.ndarray, fmt: int, sr: int) -> S.PcmTrack:
    """(frames,) or (frames, C) float signal in [-1, 1] -> interleaved PCM bytes in format fmt."""
    x = np.asarray(x, np.float64)
    if x.ndim == 1:
        x = x[:, None]
    C = x.shape[1]
    v = x.reshape(-1)
    if fmt == S.PCM_U8:
        b = (np.clip(np.round(v * 128.0), -128, 127) + 128).astype(np.uint8)
    elif fmt == S.PCM_S16:
        b = np.clip(np.round(v * 32768.0), -32768, 32767).astype("<i2").view(np.uint8)
    elif fmt == S.PCM_S24:
        q = np.clip(np.round(v * 8388608.0), -8388608, 8388607).astype("<i4").view(np.uint8).reshape(-1, 4)
        b = np.ascontiguousarray(q[:, :3]).reshape(-1)
    elif fmt == S.PCM_S32:
        b = np.clip(np.round(v * 2147483648.0), -2147483648, 2147483647).astype("<i4").view(np.uint8)
    elif fmt == S.PCM_F32:
        b = v.astype("<f4").view(np.uint8)
    else:
        b = v.astype("<f8").view(np.uint8)
    return S.PcmTrack(np.ascontiguousarray(b), fmt, C, sr)


def decode(t: S.PcmTrack) -> np.ndarray:
    """PcmTrack -> (frames, C) float32 with the device's arithmetic (all scalings are exact powers of two)."""
    d = t.data
    if t.fmt == S.PCM_U8:
        v = (d.astype(np.float32) - np.float32(128)) * np.float32(0.0078125)
    elif t.fmt == S.PCM_S16:
        v = d.view("<i2").astype(np.float32) * np.float32(2.0 ** -15)
    elif t.fmt == S.PCM_S24:
        q = d.reshape(-1, 3).astype(np.int32)
        i = q[:, 0] | (q[:, 1] << 8) | (q[:, 2] << 16)
        i = (i << 8) >> 8
        v = i.astype(np.float32) * np.float32(2.0 ** -23)
    elif t.fmt == S.PCM_S32:
        v = d.view("<i4").astype(np.float32) * np.float32(2.0 ** -31)
    elif t.fmt == S.PCM_F32:
        v = d.view("<f4").astype(np.float32)
    else:
        v = d.view("<f8").astype(np.float32)
    return v.reshape(-1, t.channels)


# ---- filters -----------------------------------------------------------------------------------------------------------
def kweight(sr: int):
    """(b, a) of the two K-weighting stages at sr, derived from the analog prototype."""
    f0, G, Q = 1681.974450955533, 3.999843853973347, 0.7071752369554196
    K = math.tan(math.pi * f0 / sr)
    Vh = 10.0 ** (G / 20.0)
    Vb = Vh ** 0.4996667741545416
    a0 = 1.0 + K / Q + K * K
    b1 = np.array([Vh + Vb * K / Q + K * K, 2.0 * (K * K - Vh), Vh - Vb * K / Q + K * K]) / a0
    a1 = np.array([1.0, 2.0 * (K * K - 1.0) / a0, (1.0 - K / Q + K * K) / a0])
    f0, Q = 38.13547087602444, 0.5003270373238773
    K = math.tan(math.pi * f0 / sr)
    d = 1.0 + K / Q + K * K
    b2 = np.array([1.0, -2.0, 1.0])
    a2 = np.array([1.0, 2.0 * (K * K - 1.0) / d, (1.0 - K / Q + K * K) / d])
    return (b1, a1), (b2, a2)


def oversampling(sr: int) -> int:
    return 4 if sr < 96000 else (2 if sr < 192000 else 1)


def taps(L: int) -> np.ndarray:
    j = np.arange(49)
    t = (j - 24) / L
    c = np.sinc(t) * 0.5 * (1.0 - np.cos(2.0 * np.pi * j / 48.0))
    c[(j - 24) % L == 0] = 0.0  # sinc at the integers: exactly 0 off centre, 1 at the centre
    c[24] = 1.0
    return c


def weights(C: int) -> np.ndarray:
    if C == 4:
        w = [1.0, 1.0, 1.41, 1.41]
    elif C == 5:
        w = [1.0, 1.0, 1.0, 1.41, 1.41]
    else:
        w = [1.0, 1.0, 1.0, 0.0, 1.41, 1.41] + [0.0] * max(0, C - 6)
    return np.array(w[:C])


def _lufs(p):
    with np.errstate(divide="ignore"):
        return -0.691 + 10.0 * np.log10(p)


def true_peak(x: np.ndarray, L: int, block: int = 1 << 22) -> float:
    """max |u| of the zero-stuffed signal convolved with the taps: u[m] = sum_j c[j] xz[m - j + 24], m < L * frames.  Long tracks
    are convolved in blocks of frames with 12 frames of context on each side (the taps reach 24 / L <= 12 frames)."""
    x = np.asarray(x, np.float64)
    frames = x.shape[0]
    c = taps(L)
    best = 0.0
    for ch in range(x.shape[1]):
        for s0 in range(0, frames, block):
            s1 = min(s0 + block, frames)
            a, b = max(0, s0 - 12), min(frames, s1 + 12)
            xz = np.zeros(L * (b - a))
            xz[::L] = x[a:b, ch]
            u = np.convolve(xz, c)[24:24 + L * (b - a)][L * (s0 - a):L * (s1 - a)]
            best = max(best, float(np.max(np.abs(u))))
    return best


def measure(t: S.PcmTrack, with_true_peak: bool = True) -> dict:
    sr = t.sample_rate
    x = decode(t).astype(np.float64)
    frames, C = x.shape
    Sb = (sr + 5) // 10
    (b1, a1), (b2, a2) = kweight(sr)
    y = lfilter(b2, a2, lfilter(b1, a1, x, axis=0), axis=0)
    nfull = frames // Sb
    e = (y[: nfull * Sb] ** 2).reshape(nfull, Sb, C).sum(axis=1)
    z = e @ weights(C)
    J, K = max(0, nfull - 3), max(0, nfull - 29)
    mom = np.array([z[j:j + 4].sum() for j in range(J)]) / (4 * Sb)
    sht = np.array([z[k:k + 30].sum() for k in range(K)]) / (30 * Sb)
    lm, ls = _lufs(mom), _lufs(sht)
    integ = -math.inf
    g = mom[lm > -70.0]
    if g.size:
        rel = _lufs(g.mean()) - 10.0
        g2 = mom[(lm > -70.0) & (lm > rel)]
        if g2.size:
            integ = float(_lufs(g2.mean()))
    lra = 0.0
    g = sht[ls > -70.0]
    if g.size:
        rel = _lufs(g.mean()) - 20.0
        v = np.sort(ls[(ls > -70.0) & (ls > rel)])
        n = v.size
        if n >= 2:
            lra = float(v[int(math.floor((n - 1) * 0.95 + 0.5))] - v[int(math.floor((n - 1) * 0.10 + 0.5))])
    sp = float(np.max(np.abs(x))) if frames else 0.0
    out = dict(integrated_lufs=integ, momentary_max_lufs=float(lm.max()) if J else -math.inf,
               short_term_max_lufs=float(ls.max()) if K else -math.inf, loudness_range_lu=lra, sample_peak=sp,
               n_momentary=J, n_short_term=K)
    if with_true_peak:
        out["true_peak"] = max(sp, true_peak(x, oversampling(sr)))
    return out
