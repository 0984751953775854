// ITU-R BS.1770-4 / EBU R128 loudness of interleaved PCM tracks (stratum_b200_loudness_batch_pcm, DESIGN §2).
//
// A track is cut into segments of S = (sr + 5) / 10 frames (100 ms, the sub-blocks of the 400 ms momentary and 3 s short-term
// windows); a work item is one (segment, channel) pair, flat over the tracks of a launch, channels of a segment adjacent.
//   pass 1  each work item runs the K-weighting cascade over its segment from zero state and keeps the end state;
//   scan    one CTA per (track, channel) turns the end states into the true start state of every segment
//           (s[k+1] = M s[k] + e[k], M = A^S computed on the host);
//   pass 2  each work item re-runs its segment from its start state and writes its sum of y^2; on the same samples it keeps the
//           sample peak and the 4x / 2x oversampled true peak (49-tap interpolator, 12 / 24 frames of context), reduced per track
//           by atomicMax on the bit pattern;
//   gate    one CTA per track: channel-weighted sub-block energies, momentary / short-term powers as in-order sums of 4 / 30
//           sub-blocks, the absolute and relative gates, the maxima and the loudness range (exact order statistics);
//   album   one CTA per album: the same gates, maxima and range over the members' momentary / short-term powers, pooled on the
//           host in ascending track order (stratum_b200_loudness_albums_pcm).
// The recurrence runs in f64: at 192 kHz the high-pass pole of stage 2 lies 1.2e-3 from the unit circle, and f32 coefficients
// and state move the 38 Hz corner by about 2 %.  The true-peak FIR runs in f32 with explicit FMAs.  No float atomics on sums:
// every result depends only on the track's own samples.
#include <math_constants.h>

#include "framed.cuh"
#include "kernels.h"
#include "pcm.cuh"

namespace sb {

// track index of flat work item w (tracks sorted by first work item)
__device__ __forceinline__ uint32_t loud_track_of(const LoudTrack* __restrict__ tr, uint32_t n, uint64_t w) {
    uint32_t lo = 0, hi = n - 1;
    while (lo < hi) {
        const uint32_t mid = (lo + hi + 1) >> 1;
        if (tr[mid].work <= w) lo = mid;
        else hi = mid - 1;
    }
    return lo;
}

struct KState {
    double z1a, z2a, z1b, z2b;
};

// One sample through the two transposed direct-form-II biquads; returns the K-weighted output.
__device__ __forceinline__ double kweight_step(const double* __restrict__ k, double x, KState& s) {
    const double y1 = __fma_rn(k[0], x, s.z1a);
    s.z1a = __fma_rn(k[1], x, __fma_rn(-k[3], y1, s.z2a));
    s.z2a = __fma_rn(k[2], x, -k[4] * y1);
    const double y2 = __fma_rn(k[5], y1, s.z1b);
    s.z1b = __fma_rn(k[6], y1, __fma_rn(-k[8], y2, s.z2b));
    s.z2b = __fma_rn(k[7], y1, -k[9] * y2);
    return y2;
}

__global__ void __launch_bounds__(256) loud_pass1_kernel(const unsigned char* __restrict__ pcm, const LoudTrack* __restrict__ tr, uint32_t n_tracks,
                                                         uint64_t n_work, double* __restrict__ st) {
    const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_work) return;
    const LoudTrack& T = tr[loud_track_of(tr, n_tracks, w)];
    const uint32_t r = (uint32_t)(w - T.work), seg = r / T.C, ch = r % T.C;
    if (seg >= T.nfull) return;  // segments past the last whole sub-block carry no energy (pass 2 still scans them for peaks)
    double k[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) k[i] = T.kw[i];
    const unsigned char* p = pcm + T.byte_off;
    KState s{0.0, 0.0, 0.0, 0.0};
    const uint64_t base = (uint64_t)seg * T.S;
    for (uint32_t i = 0; i < T.S; ++i) kweight_step(k, (double)pcm_sample(p, (base + i) * T.C + ch, T.fmt), s);
    double* o = st + 4 * w;
    o[0] = s.z1a;
    o[1] = s.z2a;
    o[2] = s.z1b;
    o[3] = s.z2b;
}

__device__ __forceinline__ void matvec4(const double* __restrict__ m, const double* v, double* out) {
#pragma unroll
    for (int i = 0; i < 4; ++i) out[i] = __fma_rn(m[4 * i], v[0], __fma_rn(m[4 * i + 1], v[1], __fma_rn(m[4 * i + 2], v[2], m[4 * i + 3] * v[3])));
}

constexpr int LOUD_SCAN_THREADS = 256;

// Exact affine scan over the segments of one (track, channel): thread t owns a run of `per` segments, composes their maps from
// zero, one thread chains the runs with M^per, then every thread replays its run from the true start and overwrites the end
// states e[k] with the start states s[k].
__global__ void __launch_bounds__(LOUD_SCAN_THREADS) loud_scan_kernel(const LoudTrack* __restrict__ tr, double* __restrict__ st) {
    const LoudTrack& T = tr[blockIdx.x];
    const uint32_t ch = blockIdx.y;
    if (ch >= T.C || T.nfull < 2) return;
    __shared__ double M[16], Mp[16], vs[LOUD_SCAN_THREADS][4];
    const uint32_t n = T.nfull;
    const uint32_t per = (n + LOUD_SCAN_THREADS - 1) / LOUD_SCAN_THREADS;
    const uint32_t a = min(threadIdx.x * per, n), b = min(a + per, n);
    if (threadIdx.x < 16) M[threadIdx.x] = T.M[threadIdx.x];
    __syncthreads();
    auto e_of = [&](uint32_t seg) { return st + 4 * (T.work + (uint64_t)seg * T.C + ch); };
    double v[4] = {0.0, 0.0, 0.0, 0.0}, t[4];
    for (uint32_t k = a; k < b; ++k) {
        const double* e = e_of(k);
        matvec4(M, v, t);
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = t[i] + e[i];
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) vs[threadIdx.x][i] = v[i];
    if (threadIdx.x == 0) {  // Mp = M^per by repeated squaring
        double r[16], q[16], tmp[16];
        for (int i = 0; i < 16; ++i) {
            r[i] = (i % 5 == 0) ? 1.0 : 0.0;
            q[i] = M[i];
        }
        for (uint32_t e = per; e; e >>= 1) {
            if (e & 1) {
                for (int i = 0; i < 4; ++i)
                    for (int j = 0; j < 4; ++j) tmp[4 * i + j] = __fma_rn(q[4 * i], r[j], __fma_rn(q[4 * i + 1], r[4 + j], __fma_rn(q[4 * i + 2], r[8 + j], q[4 * i + 3] * r[12 + j])));
                for (int i = 0; i < 16; ++i) r[i] = tmp[i];
            }
            for (int i = 0; i < 4; ++i)
                for (int j = 0; j < 4; ++j) tmp[4 * i + j] = __fma_rn(q[4 * i], q[j], __fma_rn(q[4 * i + 1], q[4 + j], __fma_rn(q[4 * i + 2], q[8 + j], q[4 * i + 3] * q[12 + j])));
            for (int i = 0; i < 16; ++i) q[i] = tmp[i];
        }
        for (int i = 0; i < 16; ++i) Mp[i] = r[i];
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // start state of every run, in order
        double s[4] = {0.0, 0.0, 0.0, 0.0};
        for (int th = 0; th < LOUD_SCAN_THREADS; ++th) {
            double nx[4];
            matvec4(Mp, s, nx);
            for (int i = 0; i < 4; ++i) {
                const double x = nx[i] + vs[th][i];
                vs[th][i] = s[i];
                s[i] = x;
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) v[i] = vs[threadIdx.x][i];
    for (uint32_t k = a; k < b; ++k) {
        double* e = e_of(k);
        matvec4(M, v, t);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const double x = t[i] + e[i];
            e[i] = v[i];
            v[i] = x;
        }
    }
}

// Pass 2 of one work item at oversampling L: frames [a, b) of channel ch, window w[k] = x[n - H + 1 + k] around the frame n the
// recurrence consumes (H = W / 2 frames of look-ahead).  Phase p of the oversampled output at n is sum_m c[p + L m] w[W-1-m].
template <int L>
__device__ __forceinline__ void loud_pass2_item(const LoudTrack& T, const unsigned char* __restrict__ p, uint32_t ch, uint64_t a, uint64_t b, bool energy,
                                                const double* k, KState& s, double& sum, float& spk, float& tpk) {
    constexpr int W = L == 1 ? 1 : 48 / L, H = W / 2;
    float c[L > 1 ? (L - 1) * W : 1];
    if constexpr (L > 1) {
#pragma unroll
        for (int ph = 1; ph < L; ++ph)
#pragma unroll
            for (int m = 0; m < W; ++m) c[(ph - 1) * W + m] = T.taps[ph + L * m];
    }
    const uint64_t frames = T.frames;
    auto x_at = [&](int64_t i) { return (i >= 0 && (uint64_t)i < frames) ? pcm_sample(p, (uint64_t)i * T.C + ch, T.fmt) : 0.0f; };
    float w[W];
#pragma unroll
    for (int j = 0; j < W; ++j) w[j] = 0.0f;
    if constexpr (L > 1)
        for (int64_t i = (int64_t)a - H + 1; i < (int64_t)a + H; ++i) {
#pragma unroll
            for (int j = 0; j + 1 < W; ++j) w[j] = w[j + 1];
            w[W - 1] = x_at(i);
        }
    for (uint64_t n = a; n < b; ++n) {
#pragma unroll
        for (int j = 0; j + 1 < W; ++j) w[j] = w[j + 1];
        w[W - 1] = x_at((int64_t)n + H);
        const float x = w[W - 1 - H];
        spk = fmaxf(spk, fabsf(x));
        if (energy) {
            const double y = kweight_step(k, (double)x, s);
            sum = __fma_rn(y, y, sum);
        }
        if constexpr (L > 1) {
#pragma unroll
            for (int ph = 1; ph < L; ++ph) {
                float u = 0.0f;
#pragma unroll
                for (int m = 0; m < W; ++m) u = __fmaf_rn(c[(ph - 1) * W + m], w[W - 1 - m], u);
                tpk = fmaxf(tpk, fabsf(u));
            }
        }
    }
}

__global__ void __launch_bounds__(256) loud_pass2_kernel(const unsigned char* __restrict__ pcm, const LoudTrack* __restrict__ tr, uint32_t n_tracks,
                                                         uint64_t n_work, const double* __restrict__ st, double* __restrict__ en, LoudOut* __restrict__ out) {
    const uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = w < n_work;
    const uint32_t t = valid ? loud_track_of(tr, n_tracks, w) : 0xffffffffu;
    float spk = 0.0f, tpk = 0.0f;
    if (valid) {
        const LoudTrack& T = tr[t];
        const uint32_t r = (uint32_t)(w - T.work), seg = r / T.C, ch = r % T.C;
        const uint64_t a = (uint64_t)seg * T.S, b = min(a + T.S, T.frames);
        const bool energy = seg < T.nfull;
        double k[10];
#pragma unroll
        for (int i = 0; i < 10; ++i) k[i] = T.kw[i];
        KState s{0.0, 0.0, 0.0, 0.0};
        if (energy && seg > 0) {
            const double* q = st + 4 * w;
            s = KState{q[0], q[1], q[2], q[3]};
        }
        double sum = 0.0;
        const unsigned char* p = pcm + T.byte_off;
        if (T.L == 4) loud_pass2_item<4>(T, p, ch, a, b, energy, k, s, sum, spk, tpk);
        else if (T.L == 2) loud_pass2_item<2>(T, p, ch, a, b, energy, k, s, sum, spk, tpk);
        else loud_pass2_item<1>(T, p, ch, a, b, energy, k, s, sum, spk, tpk);
        if (energy) en[w] = sum;
    }
    tpk = fmaxf(tpk, spk);
    // one atomic per warp when the warp lies inside one track (the common case), else one per lane
    const uint32_t t0 = __shfl_sync(0xffffffffu, t, 0);
    if (__all_sync(0xffffffffu, t == t0)) {
        for (int o = 16; o > 0; o >>= 1) {
            spk = fmaxf(spk, __shfl_xor_sync(0xffffffffu, spk, o));
            tpk = fmaxf(tpk, __shfl_xor_sync(0xffffffffu, tpk, o));
        }
        if ((threadIdx.x & 31) != 0) return;
    }
    if (valid) {  // values >= 0: bit order == value order
        atomicMax(&out[t].sample_peak_bits, __float_as_uint(spk));
        atomicMax(&out[t].true_peak_bits, __float_as_uint(tpk));
    }
}

constexpr int LOUD_GATE_THREADS = 512;

__device__ __forceinline__ double lufs_of(double power) { return -0.691 + 10.0 * log10(power); }

// In-order block sums: every thread adds its strided share in index order, then a fixed tree; the result does not depend on
// anything but the values.
__device__ __forceinline__ double block_sum_d(double v, double* sm) {
    sm[threadIdx.x] = v;
    __syncthreads();
    for (int h = LOUD_GATE_THREADS / 2; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) sm[threadIdx.x] = sm[threadIdx.x] + sm[threadIdx.x + h];
        __syncthreads();
    }
    const double r = sm[0];
    __syncthreads();
    return r;
}

__device__ __forceinline__ double block_max_d(double v, double* sm) {
    sm[threadIdx.x] = v;
    __syncthreads();
    for (int h = LOUD_GATE_THREADS / 2; h > 0; h >>= 1) {
        if ((int)threadIdx.x < h) sm[threadIdx.x] = fmax(sm[threadIdx.x], sm[threadIdx.x + h]);
        __syncthreads();
    }
    const double r = sm[0];
    __syncthreads();
    return r;
}

// Mean power of the values of pw[0..n) whose loudness lies above `gate` (and above -70 LUFS); count in *cnt.
__device__ __forceinline__ double gated_mean(const double* __restrict__ pw, uint32_t n, double gate, double* sm, double* cnt) {
    double s = 0.0, c = 0.0;
    for (uint32_t i = threadIdx.x; i < n; i += LOUD_GATE_THREADS) {
        const double l = lufs_of(pw[i]);
        if (l > -70.0 && l > gate) {
            s += pw[i];
            c += 1.0;
        }
    }
    s = block_sum_d(s, sm);
    *cnt = block_sum_d(c, sm);
    return *cnt > 0.0 ? s / *cnt : 0.0;
}

// The gates, maxima and loudness range of the momentary powers m[0..J) and short-term powers q[0..K) into o's loudness fields
// (keep: K doubles of scratch).  The per-track and the album kernel both run it on a CTA of LOUD_GATE_THREADS: the result depends
// only on the two lists, so an album of one track reproduces the track's bits.
__device__ __forceinline__ void loud_gate_lists(const double* __restrict__ m, uint32_t J, const double* __restrict__ q, uint32_t K,
                                                double* __restrict__ kp, LoudOut* __restrict__ o) {
    __shared__ double sm[LOUD_GATE_THREADS];
    __shared__ uint32_t hist[256], bcast[2], wsum[33];
    const double ninf = -CUDART_INF;
    // integrated loudness: absolute gate, then the relative gate 10 LU below the absolute-gated mean
    double cnt;
    const double abs_mean = gated_mean(m, J, ninf, sm, &cnt);
    double integrated = ninf;
    if (cnt > 0.0) {
        const double rel = lufs_of(abs_mean) - 10.0;
        const double mean = gated_mean(m, J, rel, sm, &cnt);
        if (cnt > 0.0) integrated = lufs_of(mean);
    }
    // ungated maxima
    double mx = 0.0;
    for (uint32_t j = threadIdx.x; j < J; j += LOUD_GATE_THREADS) mx = fmax(mx, m[j]);
    mx = block_max_d(mx, sm);
    double sx = 0.0;
    for (uint32_t j = threadIdx.x; j < K; j += LOUD_GATE_THREADS) sx = fmax(sx, q[j]);
    sx = block_max_d(sx, sm);
    // loudness range (EBU Tech 3342): short-term values above -70 LUFS and 20 LU below their power mean, ordered compaction,
    // then the exact 10th and 95th percentiles
    double lra = 0.0;
    const double st_mean = gated_mean(q, K, ninf, sm, &cnt);
    if (cnt > 0.0) {
        const double rel = lufs_of(st_mean) - 20.0;
        const uint32_t per = (K + LOUD_GATE_THREADS - 1) / LOUD_GATE_THREADS;
        const uint32_t a = min(threadIdx.x * per, K), b = min(a + per, K);
        uint32_t mine = 0;
        for (uint32_t j = a; j < b; ++j) {
            const double l = lufs_of(q[j]);
            mine += (l > -70.0 && l > rel) ? 1u : 0u;
        }
        uint32_t n = 0;
        uint32_t pos = block_exclusive_scan(mine, &n, wsum);
        for (uint32_t j = a; j < b; ++j) {
            const double l = lufs_of(q[j]);
            if (l > -70.0 && l > rel) kp[pos++] = q[j];
        }
        __syncthreads();
        if (n >= 2) {
            const uint32_t k10 = (uint32_t)floor((double)(n - 1) * 0.10 + 0.5), k95 = (uint32_t)floor((double)(n - 1) * 0.95 + 0.5);
            const double p10 = block_select_kth(kp, n, k10, hist, bcast);
            const double p95 = block_select_kth(kp, n, k95, hist, bcast);
            lra = lufs_of(p95) - lufs_of(p10);
        }
    }
    if (threadIdx.x == 0) {
        o->integrated = integrated;
        o->momentary_max = J > 0 ? lufs_of(mx) : ninf;
        o->short_term_max = K > 0 ? lufs_of(sx) : ninf;
        o->loudness_range = lra;
    }
}

__global__ void __launch_bounds__(LOUD_GATE_THREADS) loud_gate_kernel(const LoudTrack* __restrict__ tr, const double* __restrict__ en, double* __restrict__ zs,
                                                                      double* __restrict__ mom, double* __restrict__ sht, double* __restrict__ keep,
                                                                      LoudOut* __restrict__ out) {
    const LoudTrack& T = tr[blockIdx.x];
    if (T.nseg == 0) return;
    const uint32_t C = T.C, nfull = T.nfull, J = T.J, K = T.K;
    double* z = zs + T.seg0;
    double* m = mom + T.seg0;
    double* q = sht + T.seg0;
    for (uint32_t i = threadIdx.x; i < nfull; i += LOUD_GATE_THREADS) {
        double acc = 0.0;
        for (uint32_t c = 0; c < C; ++c) acc = acc + loud_channel_weight(C, c) * en[T.work + (uint64_t)i * C + c];
        z[i] = acc;
    }
    __syncthreads();
    const double dm = 4.0 * T.S, ds = 30.0 * T.S;
    for (uint32_t j = threadIdx.x; j < J; j += LOUD_GATE_THREADS) m[j] = (((z[j] + z[j + 1]) + z[j + 2]) + z[j + 3]) / dm;
    for (uint32_t j = threadIdx.x; j < K; j += LOUD_GATE_THREADS) {
        double acc = 0.0;
        for (int i = 0; i < 30; ++i) acc = acc + z[j + i];
        q[j] = acc / ds;
    }
    __syncthreads();
    loud_gate_lists(m, J, q, K, keep + T.seg0, out + blockIdx.x);
}

// One CTA per album over its pooled lists.
__global__ void __launch_bounds__(LOUD_GATE_THREADS) loud_album_gate_kernel(const LoudAlbum* __restrict__ al, const double* __restrict__ mom,
                                                                            const double* __restrict__ sht, double* __restrict__ keep,
                                                                            LoudOut* __restrict__ out) {
    const LoudAlbum& A = al[blockIdx.x];
    loud_gate_lists(mom + A.m0, A.J, sht + A.q0, A.K, keep + A.q0, out + blockIdx.x);
}

void launch_loud_pass1(cudaStream_t s, const void* d_pcm, const LoudTrack* d_tr, uint32_t n_tracks, uint64_t n_work, double* d_st) {
    if (n_work == 0) return;
    loud_pass1_kernel<<<(unsigned)((n_work + 255) / 256), 256, 0, s>>>(static_cast<const unsigned char*>(d_pcm), d_tr, n_tracks, n_work, d_st);
    count_launch("loudness");
}

void launch_loud_scan(cudaStream_t s, const LoudTrack* d_tr, uint32_t n_tracks, uint32_t max_channels, double* d_st) {
    if (n_tracks == 0) return;
    loud_scan_kernel<<<dim3(n_tracks, max_channels), LOUD_SCAN_THREADS, 0, s>>>(d_tr, d_st);
    count_launch("loudness");
}

void launch_loud_pass2(cudaStream_t s, const void* d_pcm, const LoudTrack* d_tr, uint32_t n_tracks, uint64_t n_work, const double* d_st, double* d_en,
                       LoudOut* d_out) {
    if (n_work == 0) return;
    loud_pass2_kernel<<<(unsigned)((n_work + 255) / 256), 256, 0, s>>>(static_cast<const unsigned char*>(d_pcm), d_tr, n_tracks, n_work, d_st, d_en, d_out);
    count_launch("loudness");
}

void launch_loud_gate(cudaStream_t s, const LoudTrack* d_tr, uint32_t n_tracks, const double* d_en, double* d_ws, uint64_t n_seg, LoudOut* d_out) {
    if (n_tracks == 0) return;
    loud_gate_kernel<<<n_tracks, LOUD_GATE_THREADS, 0, s>>>(d_tr, d_en, d_ws, d_ws + n_seg, d_ws + 2 * n_seg, d_ws + 3 * n_seg, d_out);
    count_launch("loudness");
}

void launch_loud_album_gate(cudaStream_t s, const LoudAlbum* d_al, uint32_t n_albums, const double* d_mom, const double* d_sht, double* d_keep,
                            LoudOut* d_out) {
    if (n_albums == 0) return;
    loud_album_gate_kernel<<<n_albums, LOUD_GATE_THREADS, 0, s>>>(d_al, d_mom, d_sht, d_keep, d_out);
    count_launch("loudness");
}

}  // namespace sb
