// Harmonic / percussive separation — reference features/onset/hpss.rs:71-243 (hpss_decompose) and :277-375
// (detect_hpss_onsets), used for the fourth onset detector (lib.rs:222-235) and for the percussive tempogram
// fallback (lib.rs:587-683).  On the reference's CPU path this is the worst outlier (8-9 s per 30-s clip,
// docs/progress-reports/PHASE_1F_BENCHMARKS.md:93-107).
//
// One launch per iteration.  A CTA owns a 32-frame x 32-bin tile: it stages the tile of the harmonic estimate with
// a +-margin halo in TIME and the tile of the percussive estimate with a +-margin halo in FREQUENCY in shared memory,
// every thread takes the two 21-tap medians of its elements with a 112-exchange sorting network held in registers
// (windows clipped at the spectrogram border are padded with +inf and the median index follows the valid count; an
// even count averages the two middle values, hpss.rs:197-201), applies the soft mask (hpss.rs:128-149) and writes
// the new estimates to the other half of a ping-pong pair — so the previous iterate needed by the convergence test
// (hpss.rs:152-169) is simply the buffer being read.  The per-track maximum change of an iteration is an atomicMax
// on the bit pattern; later iterations return at once for tracks that have converged.
#include "kernels.h"
#include "sortnet21.h"

namespace sb {

constexpr int HP_T = 32;       // tile: frames
constexpr int HP_B = 32;       // tile: bins
constexpr int HP_MAXM = 10;    // margin upper bound (21-wire network); larger margins are rejected by the ABI

__device__ __forceinline__ float median21(float (&v)[21], int n) {
#define CE(i, j)                    \
    {                               \
        const float a_ = v[i], b_ = v[j]; \
        v[i] = fminf(a_, b_);       \
        v[j] = fmaxf(a_, b_);       \
    }
    SORTNET21(CE)
#undef CE
    if (n == 21) return v[10];
    // clipped window: the n valid values are sorted in v[0..n), +inf above them
    const int hi = n >> 1, lo = (n & 1) ? hi : hi - 1;
    float a = 0.0f, b = 0.0f;
#pragma unroll
    for (int i = 0; i < 21; ++i) {
        a = (i == lo) ? v[i] : a;
        b = (i == hi) ? v[i] : b;
    }
    return (n & 1) ? b : (a + b) * 0.5f;
}

// converged(it): the reference breaks after iteration j >= 1 when its max change is < 1e-6
__device__ __forceinline__ bool hpss_converged_before(const TrackDev& T, int it) {
    for (int j = 1; j < it; ++j)
        if (__uint_as_float(T.hpss_maxchg[j]) < 1e-6f) return true;
    return false;
}

// nb: bins per spectrogram row (frame_size / 2 + 1)
__global__ void __launch_bounds__(256) hpss_iter_kernel(TrackDev* tr, const int32_t* __restrict__ list, float* fa, int it, uint32_t margin, int bs, int nb) {
    __shared__ float Ht[HP_T + 2 * HP_MAXM][HP_B + 1];
    __shared__ float Pt[HP_T][HP_B + 2 * HP_MAXM + 1];
    __shared__ float sred[8];
    const int t = list ? list[blockIdx.z] : blockIdx.z;
    TrackDev& T = tr[t];
    const int F = (int)T.F[bs];  // the base path's spectrogram (slot 0 unless hop_size is not 512)
    const int f0 = blockIdx.y * HP_T, b0 = blockIdx.x * HP_B;
    if (T.status != 0 || f0 >= F) return;
    if (hpss_converged_before(T, it)) return;
    const float* S = fa + T.hop[bs].spec;
    const float* Hs = it == 0 ? S : fa + T.hpss_h[it & 1];
    const float* Ps = it == 0 ? S : fa + T.hpss_p[it & 1];
    float* Hd = fa + T.hpss_h[(it + 1) & 1];
    float* Pd = fa + T.hpss_p[(it + 1) & 1];
    const int m = (int)margin;
    const float INF = __int_as_float(0x7f800000);
    // stage: harmonic rows f0-m .. f0+T+m (time halo), percussive columns b0-m .. b0+B+m (frequency halo)
    for (int i = threadIdx.x; i < (HP_T + 2 * HP_MAXM) * HP_B; i += blockDim.x) {
        const int r = i / HP_B, c = i % HP_B;
        const int f = f0 - HP_MAXM + r, b = b0 + c;
        Ht[r][c] = (f >= 0 && f < F && b < nb) ? Hs[(uint64_t)f * nb + b] : INF;
    }
    for (int i = threadIdx.x; i < HP_T * (HP_B + 2 * HP_MAXM); i += blockDim.x) {
        const int r = i / (HP_B + 2 * HP_MAXM), c = i % (HP_B + 2 * HP_MAXM);
        const int f = f0 + r, b = b0 - HP_MAXM + c;
        Pt[r][c] = (f < F && b >= 0 && b < nb) ? Ps[(uint64_t)f * nb + b] : INF;
    }
    __syncthreads();
    float mx = 0.0f;
    for (int e = threadIdx.x; e < HP_T * HP_B; e += blockDim.x) {
        const int r = e / HP_B, c = e % HP_B;
        const int f = f0 + r, b = b0 + c;
        if (f >= F || b >= nb) continue;
        float v[21];
        // time window [f-m, f+m] clipped to [0, F)
        int n = 0;
#pragma unroll
        for (int j = 0; j < 21; ++j) {
            const int d = j - HP_MAXM;
            const bool in = d >= -m && d <= m && f + d >= 0 && f + d < F;
            v[j] = in ? Ht[r + HP_MAXM + d][c] : INF;
            n += in;
        }
        const float hf = median21(v, n);
        n = 0;
#pragma unroll
        for (int j = 0; j < 21; ++j) {
            const int d = j - HP_MAXM;
            const bool in = d >= -m && d <= m && b + d >= 0 && b + d < nb;
            v[j] = in ? Pt[r][c + HP_MAXM + d] : INF;
            n += in;
        }
        const float pf = median21(v, n);
        const float original = S[(uint64_t)f * nb + b];
        const float total = hf + pf;
        float hn, pn;
        if (total > 1e-10f) {
            hn = original * (hf / total);
            pn = original * (pf / total);
        } else {
            hn = original * 0.5f;
            pn = original * 0.5f;
        }
        Hd[(uint64_t)f * nb + b] = hn;
        Pd[(uint64_t)f * nb + b] = pn;
        mx = fmaxf(mx, fmaxf(fabsf(hn - Ht[r + HP_MAXM][c]), fabsf(pn - Pt[r][c + HP_MAXM])));
    }
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) mx = fmaxf(mx, sred[w]);
        atomicMax(&T.hpss_maxchg[it], __float_as_uint(mx));  // mx >= 0: bit order == value order
    }
}

// Point the "percussive" feature slot (hop[3]) at the buffer holding the final percussive estimate.
__global__ void hpss_finish_kernel(TrackDev* tr, const int32_t* __restrict__ list, int n, int n_iter) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    TrackDev& T = tr[list ? list[i] : i];
    if (T.status != 0) return;
    int last = n_iter - 1;
    for (int j = 1; j < n_iter; ++j)
        if (__uint_as_float(T.hpss_maxchg[j]) < 1e-6f) {
            last = j;
            break;
        }
    T.hop[3].spec = T.hpss_p[(last + 1) & 1];
    T.hpss_ready = 1;
}

void launch_hpss(const WaveCtx& c, const int32_t* d_list, int n_list) {
    if (n_list == 0 || c.max_F[c.cfg.bs] == 0) return;
    const dim3 grid((c.cfg.bins + HP_B - 1) / HP_B, (c.max_F[c.cfg.bs] + HP_T - 1) / HP_T, n_list);
    for (int it = 0; it < 10; ++it) {  // DEFAULT_ITERATIONS, hpss.rs:20
        hpss_iter_kernel<<<grid, 256, 0, c.stream>>>(c.tracks, d_list, c.fa, it, c.cfg.hpss_margin, c.cfg.bs, (int)c.cfg.bins);
        count_launch("hpss");
    }
    hpss_finish_kernel<<<(n_list + 127) / 128, 128, 0, c.stream>>>(c.tracks, d_list, n_list, 10);
    count_launch("hpss");
}

}  // namespace sb
