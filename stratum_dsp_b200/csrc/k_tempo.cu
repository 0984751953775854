// Tempogram BPM estimation kernels — reference period/novelty.rs:874-986 (novelty conditioning),
// period/tempogram_fft.rs:78-192, period/tempogram_autocorr.rs:79-178, period/tempogram.rs:464-775
// (seeding, folding, scoring), lib.rs:412-545 (escalation gate and acceptance) and
// period/multi_resolution.rs:407-901 (cross-hop fusion).
#include "fft.cuh"
#include "framed.cuh"
#include "kernels.h"

namespace sb {

constexpr int FQ_E = 1, FQ_H = 2, FQ_EB = 3, FQ_HB = 6;
constexpr int PQ_SF = 1, PQ_SFB = 2, PQ_MEL = 5;
constexpr float PI_F = 3.14159265358979323846f;

__device__ __forceinline__ bool variant_on(const SrTables& st, int v) { return (st.variant_mask >> v) & 1u; }

// ---- novelty conditioning: one CTA per (variant, track) ----------------------------------------
__global__ void __launch_bounds__(256) novelty_kernel(const TrackDev* tr, const int32_t* __restrict__ list, const SrTables* srtab, const int32_t* sr_index,
                                                      int h, float* fa, DevCfg cfg) {
    __shared__ float sred[32];
    const int t = list ? list[blockIdx.y] : blockIdx.y;
    const int v = blockIdx.x;
    const TrackDev& T = tr[t];
    if (T.status != 0 || T.F[h] < 2) return;
    const SrTables& st = srtab[sr_index[t]];
    if (!variant_on(st, v)) return;
    const uint32_t L = T.F[h] - 1;
    const HopLayout& HL = T.hop[h];
    const uint64_t fm = HL.fmax;
    const float* fr = fa + HL.frame;
    const float* pr = fa + HL.pair;
    float* nov = fa + HL.nov + (uint64_t)v * fm;
    float* tmp = fa + T.scratch + (uint64_t)(2 * v) * T.fall;
    if (v == 4) {  // mel: normalised mel-SuperFlux only (novelty.rs:599-608)
        const float* s = pr + PQ_MEL * fm;
        float mx = 0.0f;
        for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) mx = fmaxf(mx, s[i]);
        mx = block_max(mx, sred);
        for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) nov[i] = mx > 1e-10f ? __fdiv_rn(s[i], mx) : s[i];
        return;
    }
    const float* sp = pr + (v == 0 ? PQ_SF : PQ_SFB + (v - 1)) * fm;
    const float* E = fr + (v == 0 ? FQ_E : FQ_EB + (v - 1)) * fm;
    const float* H = fr + (v == 0 ? FQ_H : FQ_HB + (v - 1)) * fm;
    float ms = 0.0f, me = 0.0f, mh = 0.0f;
    for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) {
        ms = fmaxf(ms, sp[i]);
        me = fmaxf(me, fmaxf(__fsub_rn(E[i + 1], E[i]), 0.0f));
        mh = fmaxf(mh, fmaxf(__fsub_rn(H[i + 1], H[i]), 0.0f));
    }
    ms = block_max(ms, sred);
    me = block_max(me, sred);
    mh = block_max(mh, sred);
    const float ws = fmaxf(cfg.nov_ws, 0.0f), we = fmaxf(cfg.nov_we, 0.0f), wh = fmaxf(cfg.nov_wh, 0.0f);
    const float wsum = fmaxf(__fadd_rn(__fadd_rn(ws, we), wh), 1e-10f);
    float mc = 0.0f;
    for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) {
        float s = sp[i];
        if (ms > 1e-10f) s = __fdiv_rn(s, ms);
        float e = fmaxf(__fsub_rn(E[i + 1], E[i]), 0.0f);
        if (me > 1e-10f) e = __fdiv_rn(e, me);
        float hh = fmaxf(__fsub_rn(H[i + 1], H[i]), 0.0f);
        if (mh > 1e-10f) hh = __fdiv_rn(hh, mh);
        float c = __fdiv_rn(__fadd_rn(__fadd_rn(__fmul_rn(s, ws), __fmul_rn(e, we)), __fmul_rn(hh, wh)), wsum);  // novelty.rs:903
        nov[i] = c;
        mc = fmaxf(mc, c);
    }
    mc = block_max(mc, sred);
    __syncthreads();
    if (mc > 1e-10f)
        for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) nov[i] = __fdiv_rn(nov[i], mc);
    __syncthreads();
    float* cur = nov;
    if (cfg.nov_lmw > 1) {  // local_mean_subtract, novelty.rs:947-967
        const uint32_t half = cfg.nov_lmw / 2;
        for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) {
            uint32_t st_ = i >= half ? i - half : 0, en = min(i + half + 1, L);
            float sum = 0.0f;
            for (uint32_t j = st_; j < en; ++j) sum = __fadd_rn(sum, cur[j]);
            float mean = __fdiv_rn(sum, (float)(en - st_));
            tmp[i] = fmaxf(__fsub_rn(cur[i], mean), 0.0f);
        }
        __syncthreads();
        cur = tmp;
    }
    float* dst = (cur == nov) ? tmp : nov;
    if (cfg.nov_smw > 1 && L >= 3) {  // smooth_moving_average_in_place, novelty.rs:970-986
        const uint32_t half = cfg.nov_smw / 2;
        for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) {
            uint32_t st_ = i >= half ? i - half : 0, en = min(i + half + 1, L);
            float sum = 0.0f;
            for (uint32_t j = st_; j < en; ++j) sum = __fadd_rn(sum, cur[j]);
            dst[i] = __fdiv_rn(sum, (float)(en - st_));
        }
        __syncthreads();
        cur = dst;
    }
    float mf = 0.0f;
    for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) mf = fmaxf(mf, cur[i]);
    mf = block_max(mf, sred);
    for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) {
        float x = cur[i];
        nov[i] = mf > 1e-10f ? __fdiv_rn(x, mf) : x;
    }
}

// ---- FFT tempogram: one CTA per (variant, track); ping-pong buffers in global memory ------------
__global__ void __launch_bounds__(512) tgfft_kernel(const TrackDev* tr, const int32_t* __restrict__ list, const SrTables* srtab, const int32_t* sr_index, int h,
                                                    float* fa) {
    __shared__ float smean;
    const int t = list ? list[blockIdx.y] : blockIdx.y;
    const int v = blockIdx.x;
    const TrackDev& T = tr[t];
    if (T.status != 0 || T.F[h] < 2) return;
    if (!variant_on(srtab[sr_index[t]], v)) return;
    const uint32_t n = T.F[h] - 1;
    const HopLayout& HL = T.hop[h];
    const float* nov = fa + HL.nov + (uint64_t)v * HL.fmax;
    const uint32_t N = next_pow2_u32(n);
    float* power = fa + HL.tgfft + (uint64_t)v * (HL.fft_cap / 2 + 1);
    if (threadIdx.x < 32) {  // mean with the reference's left-to-right f32 sum (tempogram_fft.rs:126): coalesced loads, adds in order
        const int lane = threadIdx.x;
        float s = 0.0f;
        for (uint32_t base = 0; base < n; base += 32) {
            const float v = base + lane < n ? nov[base + lane] : 0.0f;
#pragma unroll
            for (int l = 0; l < 32; ++l) s = __fadd_rn(s, __shfl_sync(0xffffffffu, v, l));  // tail lanes add +0.0 to a non-negative sum
        }
        if (lane == 0) smean = __fdiv_rn(s, (float)n);
    }
    __syncthreads();
    const float mean = smean;
    if (N < 4) {  // degenerate sizes: direct DFT of <= 2 points
        if (threadIdx.x == 0) {
            float a = n > 1 ? 0.0f : __fsub_rn(nov[0], mean);
            power[0] = __fmul_rn(a, a);
            if (N == 2) power[1] = __fmul_rn(a, a);
        }
        return;
    }
    const uint32_t M = N >> 1;
    float2* A = reinterpret_cast<float2*>(fa + HL.tgwork + (uint64_t)v * 2 * HL.fft_cap);
    float2* B = A + (HL.fft_cap >> 1);
    for (uint32_t j = threadIdx.x; j < M; j += blockDim.x) {
        float re = 0.0f, im = 0.0f;
        const uint32_t i0 = 2 * j, i1 = 2 * j + 1;
        if (i0 < n) {
            float w = 1.0f;
            if (n > 1) w = __fmul_rn(0.5f, __fsub_rn(1.0f, cosf(__fdiv_rn(__fmul_rn(__fmul_rn(2.0f, PI_F), (float)i0), (float)(n - 1)))));
            re = __fmul_rn(__fsub_rn(nov[i0], mean), w);
        }
        if (i1 < n) {
            float w = __fmul_rn(0.5f, __fsub_rn(1.0f, cosf(__fdiv_rn(__fmul_rn(__fmul_rn(2.0f, PI_F), (float)i1), (float)(n - 1)))));
            im = __fmul_rn(__fsub_rn(nov[i1], mean), w);
        }
        A[j] = make_float2(re, im);
    }
    __syncthreads();
    const uint32_t tws_n = HL.fft_cap / N;  // stride of TW_N inside the cap table
    const float2* Z = cta_cfft(A, B, HL.tgtw, M, tws_n * 2);
    for (uint32_t k = threadIdx.x; k <= M; k += blockDim.x) {
        float2 a = Z[k & (M - 1)], b = Z[(M - k) & (M - 1)];
        float2 X = rsplit(a, b, HL.tgtw[(uint64_t)k * tws_n]);
        power[k] = __fadd_rn(__fmul_rn(X.x, X.x), __fmul_rn(X.y, X.y));
    }
}

// bpm of autocorr-tempogram entry b: the reference accumulates `bpm += resolution` in f32
__device__ __forceinline__ float ac_bpm(const DevCfg& cfg, int b) {
    float bpm = cfg.min_bpm;
    for (int i = 0; i < b; ++i) bpm = __fadd_rn(bpm, cfg.bpm_resolution);
    return bpm;
}
__device__ __forceinline__ int ac_count(const DevCfg& cfg) {
    int nb = 0;
    float bpm = cfg.min_bpm;
    while (bpm <= cfg.max_bpm && nb < AC_CAP) {
        ++nb;
        bpm = __fadd_rn(bpm, cfg.bpm_resolution);
    }
    return nb;
}

// ---- autocorrelation tempogram: one thread per BPM hypothesis, sequential f32 sum -----------------
// 201 independent add chains of n terms each (tempogram_autocorr.rs:141-150): the chain latency is the
// floor, so the novelty curve is staged in shared memory (when it fits) and the loop is unrolled to
// keep the loads ahead of the adds.
constexpr uint32_t TGAC_SMEM_FLOATS = 40 * 1024;  // 160 KB: covers hop-256 curves of 6-minute tracks

// Strength of one lag: sum(nov[i] * nov[i + lag]) / (n - lag), one ordered f32 add chain (tempogram_autocorr.rs:141-150).
__device__ __forceinline__ float ac_strength(const float* nov, uint32_t n, uint32_t lag) {
    float sum = 0.0f;
    uint32_t cnt = 0;
    if (lag < n) {
        cnt = n - lag;
        const float* q = nov + lag;
        uint32_t i = 0;
        for (; i + 8 <= cnt; i += 8) {
            float pr[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) pr[u] = __fmul_rn(nov[i + u], q[i + u]);
#pragma unroll
            for (int u = 0; u < 8; ++u) sum = __fadd_rn(sum, pr[u]);
        }
        for (; i < cnt; ++i) sum = __fadd_rn(sum, __fmul_rn(nov[i], q[i]));
    }
    return cnt > 0 ? __fdiv_rn(sum, (float)cnt) : 0.0f;
}

__global__ void __launch_bounds__(256) tgac_kernel(const TrackDev* tr, const int32_t* __restrict__ list, const SrTables* srtab, const int32_t* sr_index, int h,
                                                   float* fa, DevCfg cfg, uint32_t smem_floats) {
    extern __shared__ float snov[];
    const int t = list ? list[blockIdx.y] : blockIdx.y;
    const int v = blockIdx.x;
    const TrackDev& T = tr[t];
    if (T.status != 0 || T.F[h] < 2) return;
    if (!variant_on(srtab[sr_index[t]], v)) return;
    const uint32_t n = T.F[h] - 1;
    const HopLayout& HL = T.hop[h];
    const float* gnov = fa + HL.nov + (uint64_t)v * HL.fmax;
    const float* nov = gnov;
    if (n <= smem_floats) {
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) snov[i] = gnov[i];
        nov = snov;
    }
    __syncthreads();
    float* ac = fa + HL.tgac + (uint64_t)v * AC_CAP;
    const int nb = ac_count(cfg);
    const float frame_rate = __fdiv_rn((float)T.sr, (float)HL.hop);
    for (int b = threadIdx.x; b < nb; b += blockDim.x) {
        const float bpm = ac_bpm(cfg, b);
        const float fpb = __fdiv_rn(frame_rate, __fdiv_rn(bpm, 60.0f));
        ac[b] = ac_strength(nov, n, as_u32(fpb));
    }
}

// ---- autocorrelation tempogram of a fine BPM grid: one add chain per distinct lag ----------------------------------------
// A hypothesis enters the strength only through lag = trunc(frame_rate / (bpm / 60)), which does not increase along the grid, so
// equal lags form contiguous runs: 40..240 BPM at hop 512 and 44.1 kHz has at most 109 of them whatever the resolution.  Pass 1
// walks the grid 256 hypotheses at a time, compacts the run heads in order (block scan of the head flags) and computes one chain
// per run, up to 256 runs at a time; run r's strength is stored at ac[r] (r <= the run's first index).  Pass 2 walks the grid
// from the top down and copies ac[run(b)] to ac[b]: every ac[r] it reads still holds a run strength.  Each strength is the
// chain tgac_kernel computes for the same lag, so the result is bit-identical to the per-hypothesis form.
__global__ void __launch_bounds__(256) tgac_lag_kernel(const TrackDev* tr, const int32_t* __restrict__ list, const SrTables* srtab, const int32_t* sr_index,
                                                       int h, float* fa, DevCfg cfg, uint32_t smem_floats) {
    extern __shared__ float snov[];
    __shared__ uint32_t pend[512];  // lags of the runs found and not computed yet (< 256 carried over + <= 256 new)
    __shared__ uint32_t wsum[33];
    const int t = list ? list[blockIdx.y] : blockIdx.y;
    const int v = blockIdx.x;
    const TrackDev& T = tr[t];
    if (T.status != 0 || T.F[h] < 2) return;
    if (!variant_on(srtab[sr_index[t]], v)) return;
    const uint32_t n = T.F[h] - 1;
    const HopLayout& HL = T.hop[h];
    const float* gnov = fa + HL.nov + (uint64_t)v * HL.fmax;
    const float* nov = gnov;
    if (n <= smem_floats) {
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) snov[i] = gnov[i];
        nov = snov;
    }
    __syncthreads();
    float* ac = fa + HL.tgac + (uint64_t)v * cfg.ac_stride;
    const uint32_t nb = cfg.n_bpm, B = blockDim.x;
    const float frame_rate = __fdiv_rn((float)T.sr, (float)HL.hop);
    auto lag_of = [&](uint32_t b) { return as_u32(__fdiv_rn(frame_rate, __fdiv_rn(cfg.bpm_tab[b], 60.0f))); };
    auto is_head = [&](uint32_t b) { return b < nb && (b == 0 || lag_of(b) != lag_of(b - 1)); };
    uint32_t n_pend = 0, n_runs = 0;  // block-uniform
    for (uint32_t c0 = 0; c0 < nb; c0 += B) {
        const uint32_t b = c0 + threadIdx.x;
        const bool head = is_head(b);
        uint32_t tot;
        const uint32_t pos = block_exclusive_scan(head ? 1u : 0u, &tot, wsum);
        if (head) pend[n_pend + pos] = lag_of(b);
        n_pend += tot;
        __syncthreads();
        const bool last = c0 + B >= nb;
        while (n_pend >= B || (last && n_pend > 0)) {
            const uint32_t m = min(n_pend, B);
            if (threadIdx.x < m) ac[n_runs + threadIdx.x] = ac_strength(nov, n, pend[threadIdx.x]);
            const bool carry = threadIdx.x + m < n_pend;  // n_pend - m < B
            const uint32_t kept = carry ? pend[threadIdx.x + m] : 0u;
            __syncthreads();
            if (carry) pend[threadIdx.x] = kept;
            __syncthreads();
            n_runs += m;
            n_pend -= m;
        }
    }
    uint32_t above = 0;  // run heads at or above the end of the current chunk
    for (int64_t c0 = (int64_t)((nb - 1) / B) * B; c0 >= 0; c0 -= B) {
        const uint32_t b = (uint32_t)c0 + threadIdx.x;
        const bool head = is_head(b);
        uint32_t tot;
        const uint32_t before = block_exclusive_scan(head ? 1u : 0u, &tot, wsum);  // heads in [c0, b)
        const float x = b < nb ? ac[n_runs - above - tot + before + (head ? 1u : 0u) - 1u] : 0.0f;
        __syncthreads();
        if (b < nb) ac[b] = x;
        __syncthreads();
        above += tot;
    }
}

// ---- candidate seeding / scoring: one CTA per track --------------------------------------------
struct FftList {
    const float* p;  // power, all bins
    uint32_t kmin, kmax;  // inclusive range of bins with bpm in [min,max]; kmin > kmax = empty
    float res;            // frame_rate / fft_size
};
__device__ __forceinline__ float fft_bpm(const FftList& l, uint32_t k) { return __fmul_rn(__fmul_rn((float)k, l.res), 60.0f); }

// lookup_nearest over the power-sorted FFT list (tempogram.rs:518-529): nearest bpm within tol;
// ties resolved by list order = (power desc, bin asc).
__device__ inline float lookup_fft(const FftList& l, float bpm, float tol) {
    if (l.kmin > l.kmax) return 0.0f;
    float kf = __fdiv_rn(bpm, __fmul_rn(l.res, 60.0f));
    int kc = (int)kf;
    float best_d = INFINITY, best_v = 0.0f;
    int lo = max(kc - 3, (int)l.kmin), hi = min(kc + 3, (int)l.kmax);
    for (int k = lo; k <= hi; ++k) {
        float d = fabsf(__fsub_rn(fft_bpm(l, (uint32_t)k), bpm));
        if (!(d <= tol)) continue;
        float v = l.p[k];
        if (d < best_d || (d == best_d && v > best_v)) {
            best_d = d;
            best_v = v;
        }
    }
    return best_v;
}

// lookup_nearest over the strength-sorted autocorrelation list (tempogram.rs:518-529), ties by strength.  acb[b] = bpm of entry b.
// Coarse grids: entry b sits within +-3 steps of (bpm - min) / res.  Fine grids: the accumulated values drift from min + b * res (5 steps
// at 0.01 BPM over 40..240), so the entry is found by value: the lower bound of bpm in the strictly increasing table and its left
// neighbour are the two nearest entries.
template <bool FINE>
__device__ inline float lookup_ac(const float* ac, int nb, const DevCfg& cfg, const float* acb, float bpm, float tol) {
    int lo, hi;
    if constexpr (FINE) {
        int a = 0, e = nb;
        while (a < e) {
            const int mid = (a + e) >> 1;
            if (acb[mid] < bpm) a = mid + 1;
            else e = mid;
        }
        lo = max(a - 1, 0);
        hi = min(a, nb - 1);
    } else {
        float bf = __fdiv_rn(__fsub_rn(bpm, cfg.min_bpm), cfg.bpm_resolution);
        int bc = (int)bf;
        lo = max(bc - 3, 0);
        hi = min(bc + 3, nb - 1);
    }
    float best_d = INFINITY, best_v = 0.0f;
    for (int b = lo; b <= hi; ++b) {
        float d = fabsf(__fsub_rn(acb[b], bpm));
        if (!(d <= tol)) continue;
        float v = ac[b];
        if (d < best_d || (d == best_d && v > best_v)) {
            best_d = d;
            best_v = v;
        }
    }
    return best_v;
}

template <bool FINE>  // FINE: more than AC_CAP hypotheses, read from the device table cfg.bpm_tab
__global__ void __launch_bounds__(256) score_kernel(TrackDev* tr, const int32_t* __restrict__ list, const SrTables* srtab, const int32_t* sr_index, int h,
                                                    float* fa, DevCfg cfg, uint32_t top_n) {
    __shared__ float sval[8];
    __shared__ int sidx[8];
    __shared__ int top_fft[MAX_VARIANTS][8], top_ac[MAX_VARIANTS][8];
    __shared__ int ntop_fft[MAX_VARIANTS], ntop_ac[MAX_VARIANTS];
    __shared__ float cand[MAX_CANDS], sorted[MAX_CANDS];
    __shared__ float sc_score[MAX_CANDS], sc_fft[MAX_CANDS], sc_ac[MAX_CANDS];
    __shared__ int order[MAX_CANDS];
    __shared__ int n_cand, n_uniq;
    __shared__ float acb[AC_CAP];  // bpm of autocorr entry b, accumulated like the reference's `bpm += resolution`
    const int t = list ? list[blockIdx.x] : blockIdx.x;
    TrackDev& T = tr[t];
    if (threadIdx.x == 0) {
        if constexpr (!FINE) {
            float bq = cfg.min_bpm;
            for (int b = 0; b < AC_CAP; ++b) { acb[b] = bq; bq = __fadd_rn(bq, cfg.bpm_resolution); }
        }
        T.est[h].ok = 0;
        T.est[h].n_cands = 0;
    }
    if (T.status != 0 || T.F[h] < 2) return;
    const SrTables& st = srtab[sr_index[t]];
    const HopLayout& HL = T.hop[h];
    const uint32_t n = T.F[h] - 1;
    const uint32_t N = next_pow2_u32(n);
    const float frame_rate = __fdiv_rn((float)T.sr, (float)HL.hop);
    FftList fl[MAX_VARIANTS];
    const float res = __fdiv_rn(frame_rate, (float)N);
    // bins with bpm in range: bpm(k) is monotone in k, find the inclusive range by scanning from estimates
    uint32_t kmin, kmax;
    {
        const uint32_t half = N / 2;
        FftList tmp{nullptr, 0, half, res};
        uint32_t a = (uint32_t)fmaxf(floorf(__fdiv_rn(cfg.min_bpm, __fmul_rn(res, 60.0f))) - 2.0f, 0.0f);
        while (a <= half && !(fft_bpm(tmp, a) >= cfg.min_bpm)) ++a;
        uint32_t b = min((uint32_t)(__fdiv_rn(cfg.max_bpm, __fmul_rn(res, 60.0f))) + 2u, half);
        while (b > 0 && !(fft_bpm(tmp, b) <= cfg.max_bpm)) --b;
        if (!(fft_bpm(tmp, b) <= cfg.max_bpm)) { a = 1; b = 0; }
        kmin = a;
        kmax = b;
    }
    const int nb = FINE ? (int)cfg.n_bpm : ac_count(cfg);
    const float* bt = FINE ? cfg.bpm_tab : acb;
    const uint64_t acs = FINE ? cfg.ac_stride : AC_CAP;
    for (int v = 0; v < MAX_VARIANTS; ++v) {
        fl[v].p = fa + HL.tgfft + (uint64_t)v * (HL.fft_cap / 2 + 1);
        fl[v].kmin = kmin;
        fl[v].kmax = kmax;
        fl[v].res = res;
    }
    // top-8 per list (tempogram.rs:538-542)
    for (int v = 0; v < MAX_VARIANTS; ++v) {
        if (!variant_on(st, v)) {
            if (threadIdx.x == 0) { ntop_fft[v] = 0; ntop_ac[v] = 0; }
            continue;
        }
        const float* pf = fl[v].p;
        const float* pa = fa + HL.tgac + (uint64_t)v * acs;
        int c1 = (kmin <= kmax) ? block_topk<8>([&](int i) { return pf[i]; }, (int)kmin, (int)kmax, top_fft[v], sval, sidx) : 0;
        int c2 = block_topk<8>([&](int i) { return pa[i]; }, 0, nb - 1, top_ac[v], sval, sidx);
        if (threadIdx.x == 0) { ntop_fft[v] = c1; ntop_ac[v] = c2; }
    }
    __syncthreads();
    const float fft_primary = ntop_fft[0] > 0 ? fft_bpm(fl[0], (uint32_t)top_fft[0][0]) : 0.0f;
    const float ac_primary = ntop_ac[0] > 0 ? bt[top_ac[0][0]] : 0.0f;
    if (threadIdx.x == 0) {
        const float FACT[7] = {1.0f, 0.5f, 2.0f, 1.0f / 3.0f, 3.0f, 2.0f / 3.0f, 3.0f / 2.0f};
        int c = 0;
        auto push = [&](float base) {
            for (int f = 0; f < 7; ++f) {
                float b = __fmul_rn(base, FACT[f]);
                if (isfinite(b) && b >= cfg.min_bpm && b <= cfg.max_bpm && c < MAX_CANDS) cand[c++] = b;
            }
        };
        for (int v = 0; v < MAX_VARIANTS; ++v) {
            if (!variant_on(st, v)) continue;
            for (int i = 0; i < ntop_fft[v]; ++i) push(fft_bpm(fl[v], (uint32_t)top_fft[v][i]));
            for (int i = 0; i < ntop_ac[v]; ++i) push(bt[top_ac[v][i]]);
        }
        if (fft_primary > 0.0f) push(fft_primary);
        if (ac_primary > 0.0f) push(ac_primary);
        n_cand = c;
    }
    __syncthreads();
    const int nc = n_cand;
    // ascending rank sort
    for (int i = threadIdx.x; i < nc; i += blockDim.x) {
        float x = cand[i];
        int r = 0;
        for (int j = 0; j < nc; ++j) r += (cand[j] < x) || (cand[j] == x && j < i);
        sorted[r] = x;
    }
    __syncthreads();
    if (threadIdx.x == 0) {  // cluster within 0.75 BPM (tempogram.rs:561-570)
        int u = 0;
        for (int i = 0; i < nc; ++i) {
            if (u > 0 && fabsf(__fsub_rn(sorted[i], cand[u - 1])) < 0.75f) continue;
            cand[u++] = sorted[i];  // cand[] reused as uniq[] (u <= i always)
        }
        n_uniq = u;
    }
    __syncthreads();
    const int nu = n_uniq;
    const float ac_tol = fmaxf(cfg.bpm_resolution, 0.5f);
    const float support_thr = clamp_rs(cfg.support_thr, 0.0f, 1.0f);
    const float bonus = fmaxf(cfg.consensus_bonus, 0.0f);
    // scoring variants (tempogram.rs:464-484): seed_only -> the full-band variant alone; otherwise every active variant, weighted,
    // in the reference's order full, low, mid, high, mel
    const float vw[MAX_VARIANTS] = {cfg.w_full, cfg.w_low, cfg.w_mid, cfg.w_high, cfg.w_mel};
    const int n_score = cfg.seed_only ? 1 : MAX_VARIANTS;
    float vmax_fft[MAX_VARIANTS], vmax_ac[MAX_VARIANTS];
    float w_sum = 0.0f;
    for (int v = 0; v < n_score; ++v) {
        vmax_fft[v] = vmax_ac[v] = 1.0f;
        if (!variant_on(st, v)) continue;
        const float* acv = fa + HL.tgac + (uint64_t)v * acs;
        vmax_fft[v] = fmaxf(ntop_fft[v] > 0 ? fl[v].p[top_fft[v][0]] : 1.0f, 1e-12f);
        vmax_ac[v] = fmaxf(ntop_ac[v] > 0 ? acv[top_ac[v][0]] : 1.0f, 1e-12f);
        w_sum = __fadd_rn(w_sum, fmaxf(vw[v], 0.0f));
    }
    w_sum = fmaxf(w_sum, 1e-6f);
    for (int i = threadIdx.x; i < nu; i += blockDim.x) {
        const float bpm = cand[i];
        float fft_acc = 0.0f, ac_acc = 0.0f;
        for (int v = 0; v < n_score; ++v) {
            if (!variant_on(st, v) || !(vw[v] > 0.0f)) continue;
            const float* acv = fa + HL.tgac + (uint64_t)v * acs;
            float fv = lookup_fft(fl[v], bpm, 0.75f);
            float av = lookup_ac<FINE>(acv, nb, cfg, bt, bpm, ac_tol);
            fft_acc = __fadd_rn(fft_acc, __fmul_rn(vw[v], clamp_rs(__fdiv_rn(fv, vmax_fft[v]), 0.0f, 1.0f)));
            ac_acc = __fadd_rn(ac_acc, __fmul_rn(vw[v], clamp_rs(__fdiv_rn(av, vmax_ac[v]), 0.0f, 1.0f)));
        }
        const float fft_norm = clamp_rs(__fdiv_rn(fft_acc, w_sum), 0.0f, 1.0f);
        const float ac_norm = clamp_rs(__fdiv_rn(ac_acc, w_sum), 0.0f, 1.0f);
        float score = __fadd_rn(__fmul_rn(0.55f, ac_norm), __fmul_rn(0.45f, fft_norm));
        if (bonus > 0.0f && (cfg.band_fusion || cfg.mel_enabled)) {
            uint32_t support = 0;
            for (int v = 1; v < MAX_VARIANTS; ++v) {
                if (!variant_on(st, v)) continue;
                const float* acv = fa + HL.tgac + (uint64_t)v * acs;
                const float mf = fmaxf(ntop_fft[v] > 0 ? fl[v].p[top_fft[v][0]] : 1.0f, 1e-12f);
                const float ma = fmaxf(ntop_ac[v] > 0 ? acv[top_ac[v][0]] : 1.0f, 1e-12f);
                float sf = clamp_rs(__fdiv_rn(lookup_fft(fl[v], bpm, 0.75f), mf), 0.0f, 1.0f);
                float sa = clamp_rs(__fdiv_rn(lookup_ac<FINE>(acv, nb, cfg, bt, bpm, ac_tol), ma), 0.0f, 1.0f);
                if (fmaxf(sf, sa) >= support_thr) ++support;
            }
            if (support >= 2) score = __fmul_rn(score, __fadd_rn(1.0f, __fmul_rn(bonus, __fsub_rn((float)support, 1.0f))));
        }
        if (bpm > 180.0f) score = __fmul_rn(score, 0.80f);
        else if (bpm < 60.0f) score = __fmul_rn(score, 0.90f);
        sc_score[i] = score;
        sc_fft[i] = fft_norm;
        sc_ac[i] = ac_norm;
    }
    __syncthreads();
    // stable sort by score desc (tempogram.rs:655-659)
    for (int i = threadIdx.x; i < nu; i += blockDim.x) {
        float x = sc_score[i];
        int r = 0;
        for (int j = 0; j < nu; ++j) r += (sc_score[j] > x) || (sc_score[j] == x && j < i);
        order[r] = i;
    }
    __syncthreads();
    if (threadIdx.x == 0 && nu > 0) {
        int bi = order[0];
        if (cand[bi] > 180.0f) {  // tempo-octave fold (tempogram.rs:669-699)
            float folded = __fdiv_rn(cand[bi], 2.0f);
            if (folded >= cfg.min_bpm && folded <= cfg.max_bpm) {
                for (int r = 0; r < nu; ++r) {
                    int j = order[r];
                    if (fabsf(__fsub_rn(cand[j], folded)) < 0.75f) {
                        const float eps = 1e-6f;
                        float ar = __fdiv_rn(__fadd_rn(sc_ac[bi], eps), __fadd_rn(sc_ac[j], eps));
                        float frr = __fdiv_rn(__fadd_rn(sc_fft[bi], eps), __fadd_rn(sc_fft[j], eps));
                        if (!(ar > 2.0f && frr > 2.0f)) bi = j;
                        break;
                    }
                }
            }
        }
        const float best_score = sc_score[bi], best_bpm = cand[bi];
        float conf = 0.0f;
        if (best_score > 1e-12f) {
            float second = nu > 1 ? sc_score[order[1]] : 0.0f;
            conf = clamp_rs(__fdiv_rn(fmaxf(__fsub_rn(best_score, second), 0.0f), best_score), 0.0f, 1.0f);
        }
        uint32_t agree = 0;
        if (fft_primary > 0.0f && fabsf(__fsub_rn(fft_primary, best_bpm)) < 2.0f) ++agree;
        if (ac_primary > 0.0f && fabsf(__fsub_rn(ac_primary, best_bpm)) < 2.0f) ++agree;
        T.est[h].bpm = best_bpm;
        T.est[h].confidence = conf;
        T.est[h].agreement = agree;
        T.est[h].ok = 1;
        T.est[h].n_cands = min((uint32_t)nu, top_n);
    }
    __syncthreads();
    if (nu > 0) {
        TempoCandDev* out = reinterpret_cast<TempoCandDev*>(fa + T.cands[h]);
        const int keep = min((uint32_t)nu, top_n);
        for (int r = threadIdx.x; r < keep; r += blockDim.x) {
            int j = order[r];
            out[r] = TempoCandDev{cand[j], sc_score[j], sc_fft[j], sc_ac[j]};
        }
    }
}

// ---- escalation gate (lib.rs:412-459) ----------------------------------------------------------
__device__ inline float cand_support(const TempoCandDev* c, uint32_t n, float bpm, float tol) {
    float best = 0.0f;
    for (uint32_t i = 0; i < n; ++i)
        if (fabsf(__fsub_rn(c[i].bpm, bpm)) <= tol) best = fmaxf(best, c[i].score);
    return best;
}

__global__ void escalation_gate_kernel(TrackDev* tr, const float* fa, int n_tracks, DevCfg cfg) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tracks) return;
    TrackDev& T = tr[t];
    T.escalate = 0;
    T.mr_triggered = -1;
    T.mr_used = -1;
    T.perc_triggered = -1;
    T.perc_used = -1;
    T.chosen_agree = T.est[cfg.bs].ok ? T.est[cfg.bs].agreement : 0;
    T.trap_low = T.trap_high = 0;
    if (T.status != 0 || !T.est[cfg.bs].ok || !cfg.mr_enabled || cfg.force_legacy) return;
    const TempoEstDev& b = T.est[cfg.bs];  // the base estimate (slot 0 unless hop_size is not 512)
    const TempoCandDev* c = reinterpret_cast<const TempoCandDev*>(fa + T.cands[cfg.bs]);
    const bool trap_low = b.bpm >= 55.0f && b.bpm <= 80.0f;
    const bool trap_high = b.bpm >= 170.0f && b.bpm <= 200.0f;
    const float tol = fmaxf(2.0f, cfg.bpm_resolution);
    const float s_base = cand_support(c, b.n_cands, b.bpm, tol);
    const float s_2x = cand_support(c, b.n_cands, __fmul_rn(b.bpm, 2.0f), tol);
    const float s_half = cand_support(c, b.n_cands, __fmul_rn(b.bpm, 0.5f), tol);
    const bool family = (s_2x > 0.0f && s_2x >= __fmul_rn(s_base, 0.90f)) || (s_half > 0.0f && s_half >= __fmul_rn(s_base, 0.90f));
    const float b2 = __fmul_rn(b.bpm, 2.0f);
    const bool fold_into_trap = b2 >= 170.0f && b2 <= 200.0f;
    const bool weak = b.agreement == 0 || b.confidence < 0.06f;
    const bool ambiguous = trap_low || trap_high || family || (weak && fold_into_trap);
    T.escalate = ambiguous ? 1 : 0;
    T.mr_triggered = ambiguous ? 1 : 0;
    T.mr_used = 0;
    T.perc_triggered = (ambiguous && trap_low) ? 1 : 0;
    if (cfg.perc_fallback) T.perc_used = 0;  // lib.rs:587-683: Some(false) unless the fallback is evaluated and accepted
    T.trap_low = trap_low;
    T.trap_high = trap_high;
}

// ---- escalation list (lib.rs:412-459): ordered compaction of the gate's flags, on the device ---------------------------
// list[0 .. count) = indices of the escalated tracks in ascending order, *count_out = count.  The hop-256 / hop-1024 work
// areas of an escalated track live in arena slots of `slot_stride` floats starting at `slot_base`; the host planned their
// layouts relative to the slot start (engine.cu: plan_escalation), so the track at list position p only has its offsets moved
// to slot p mod n_slots.  Replaces a read-back of every track record plus two small copies per escalated track; the host
// reads one integer.  One CTA; tracks are taken 1024 at a time.
__global__ void __launch_bounds__(1024) escalation_compact_kernel(TrackDev* tr, int n_tracks, int32_t* list, int32_t* count_out, uint64_t slot_base,
                                                                  uint64_t slot_stride, uint32_t n_slots) {
    __shared__ int wcnt[32];
    __shared__ int base_s;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    if (tid == 0) base_s = 0;
    __syncthreads();
    for (int c0 = 0; c0 < n_tracks; c0 += 1024) {
        const int t = c0 + tid;
        const bool flag = t < n_tracks && tr[t].status == 0 && tr[t].escalate != 0;
        const uint32_t m = __ballot_sync(0xffffffffu, flag);
        if (lane == 0) wcnt[wid] = __popc(m);
        __syncthreads();
        int before = base_s;
        for (int q = 0; q < wid; ++q) before += wcnt[q];
        if (flag) {
            const int pos = before + __popc(m & ((1u << lane) - 1u));
            list[pos] = t;
            const uint64_t add = slot_base + (uint64_t)((uint32_t)pos % n_slots) * slot_stride;
            TrackDev& T = tr[t];
            for (int h = 1; h <= 2; ++h) {
                HopLayout& H = T.hop[h];
                H.spec += add;
                H.frame += add;
                H.pair += add;
                H.nov += add;
                H.tgfft += add;
                H.tgac += add;
                H.tgwork += add;
                T.cands[h] += add;
            }
        }
        __syncthreads();
        if (tid == 0) {
            int tot = 0;
            for (int q = 0; q < 32; ++q) tot += wcnt[q];
            base_s += tot;
        }
        __syncthreads();
    }
    if (tid == 0) *count_out = base_s;
}

// ---- multi-resolution fusion (multi_resolution.rs:407-901): one CTA per escalated track ----------
__device__ inline float mr_lookup(const TempoCandDev* c, uint32_t n, float bpm, float tol) {  // :282-293
    float best_d = INFINITY, best_s = 0.0f;
    for (uint32_t i = 0; i < n; ++i) {
        float d = fabsf(__fsub_rn(c[i].bpm, bpm));
        if (d <= tol && d < best_d) {
            best_d = d;
            best_s = c[i].score;
        }
    }
    return best_s;
}

// beat_contrast_score (:580-678) — block collective: phases are spread over threads, each phase
// accumulates in beat order; the max over phases is order-free.
__device__ inline float block_beat_contrast(const float* nov, uint32_t n, float total, uint32_t sr, uint32_t hop, float bpm, float* sred) {
    if (n < 16 || !(isfinite(bpm) && bpm > 0.0f) || sr == 0 || hop == 0) return 0.0f;
    const float fpb = __fdiv_rn(__fmul_rn(60.0f, (float)sr), __fmul_rn(bpm, (float)hop));
    if (!isfinite(fpb) || fpb < 3.0f) return 0.0f;
    const int per = as_i32(roundf(fpb));
    if (per < 3 || per > 512) return 0.0f;
    const uint32_t period = (uint32_t)per, w = 2;
    auto win_max = [&](uint32_t c) {
        uint32_t st = c >= w ? c - w : 0, en = min(c + w + 1, n);
        float mx = 0.0f;
        for (uint32_t j = st; j < en; ++j) mx = fmaxf(mx, nov[j]);
        return mx;
    };
    const float denom = fmaxf(__fdiv_rn(total, (float)n), 1e-6f);
    float best = -1e9f;
    for (uint32_t phase = threadIdx.x; phase < period; phase += blockDim.x) {
        float bs = 0.0f, hs = 0.0f, ts = 0.0f;
        uint32_t bn = 0, hn = 0, tn = 0;
        for (uint32_t i = phase; i < n; i += period) {
            bs = __fadd_rn(bs, win_max(i));
            ++bn;
            if (period >= 6) {
                uint32_t j = i + period / 2;
                if (j < n) { hs = __fadd_rn(hs, win_max(j)); ++hn; }
            }
            if (period >= 9) {
                for (uint32_t frac = 1; frac <= 2; ++frac) {
                    uint32_t j = i + (period * frac) / 3;
                    if (j < n) { ts = __fadd_rn(ts, win_max(j)); ++tn; }
                }
            }
        }
        float bm = bn ? __fdiv_rn(bs, (float)bn) : 0.0f, hm = hn ? __fdiv_rn(hs, (float)hn) : 0.0f, tm = tn ? __fdiv_rn(ts, (float)tn) : 0.0f;
        float contrast = __fsub_rn(__fsub_rn(bm, __fmul_rn(0.60f, hm)), __fmul_rn(0.40f, tm));
        float score = clamp_rs(__fdiv_rn(contrast, denom), -10.0f, 10.0f);
        best = fmaxf(best, score);
    }
    // block max (values may be negative: cannot use block_max's zero identity)
    for (int o = 16; o > 0; o >>= 1) best = fmaxf(best, __shfl_xor_sync(0xffffffffu, best, o));
    if ((threadIdx.x & 31) == 0) sred[threadIdx.x >> 5] = best;
    __syncthreads();
    float r = -1e9f;
    for (int w2 = 0; w2 < (int)(blockDim.x >> 5); ++w2) r = fmaxf(r, sred[w2]);
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(128) multires_fusion_kernel(TrackDev* tr, const int32_t* __restrict__ list, const float* fa, DevCfg cfg) {
    __shared__ float sred[32];
    __shared__ float fam_bpm[6], fam_support[6], fam_align[6];
    __shared__ int n_fam, run_family;
    __shared__ float s_total, best_bpm_s, best_score_s, second_s;
    __shared__ int mr_ok;
    const int t = list[blockIdx.x];
    TrackDev& T = tr[t];
    const TempoCandDev* c512 = reinterpret_cast<const TempoCandDev*>(fa + T.cands[0]);
    const TempoCandDev* c256 = reinterpret_cast<const TempoCandDev*>(fa + T.cands[1]);
    const TempoCandDev* c1024 = reinterpret_cast<const TempoCandDev*>(fa + T.cands[2]);
    const uint32_t top_k = max(cfg.mr_top_k, 1u);
    const uint32_t n512 = min(T.est[0].n_cands, top_k), n256 = T.est[1].n_cands, n1024 = T.est[2].n_cands;
    const float tol = fmaxf(2.0f, cfg.bpm_resolution);
    const float* nov = fa + T.hop[0].nov;  // full-band hop-512 novelty (multi_resolution.rs:681-695 recomputes the same curve)
    const uint32_t nn = T.F[0] >= 1 ? T.F[0] - 1 : 0;
    auto total_support = [&](float bpm, uint32_t* agree) {
        float a = mr_lookup(c256, n256, bpm, tol), b = mr_lookup(c512, n512, bpm, tol), d = mr_lookup(c1024, n1024, bpm, tol);
        *agree = (a > 0.0f) + (b > 0.0f) + (d > 0.0f);
        return __fadd_rn(__fadd_rn(a, b), d);
    };
    if (threadIdx.x == 0) {
        mr_ok = 0;
        run_family = 0;
        n_fam = 0;
        if (T.est[0].ok && T.est[1].ok && T.est[2].ok) {
            // hypotheses (:407-523)
            float hb[32], hs[32];
            int nh = 0;
            const float w512 = cfg.mr_w512, w256 = cfg.mr_w256, w1024 = cfg.mr_w1024, dt = cfg.mr_dt;
            for (uint32_t ti = 0; ti < n512 && nh < 32; ++ti) {
                const float tb = c512[ti].bpm;
                if (!(isfinite(tb) && tb > 0.0f)) continue;
                const float t2 = __fmul_rn(tb, 2.0f), th = __fmul_rn(tb, 0.5f);
                float s_t_512 = mr_lookup(c512, n512, tb, tol), s_t_256 = mr_lookup(c256, n256, tb, tol), s_t_1024 = mr_lookup(c1024, n1024, tb, tol);
                float s_2_512 = mr_lookup(c512, n512, t2, tol), s_2_256 = mr_lookup(c256, n256, t2, tol), s_2_1024 = mr_lookup(c1024, n1024, t2, tol);
                float s_h_512 = mr_lookup(c512, n512, th, tol), s_h_256 = mr_lookup(c256, n256, th, tol), s_h_1024 = mr_lookup(c1024, n1024, th, tol);
                float h_t = __fadd_rn(__fadd_rn(__fmul_rn(w512, s_t_512), __fmul_rn(w256, s_t_256)), __fmul_rn(w1024, s_t_1024));
                const float omdt = __fsub_rn(1.0f, dt);
                float h_2t = __fadd_rn(__fadd_rn(__fmul_rn(w512, __fadd_rn(__fmul_rn(dt, s_t_512), __fmul_rn(omdt, s_2_512))), __fmul_rn(w256, s_2_256)),
                                       __fmul_rn(w1024, s_2_1024));
                float h_half = __fadd_rn(__fadd_rn(__fmul_rn(w512, __fadd_rn(__fmul_rn(dt, s_t_512), __fmul_rn(omdt, s_h_512))), __fmul_rn(w256, s_h_256)),
                                         __fmul_rn(w1024, s_h_1024));
                if (s_t_1024 > __fmul_rn(s_h_1024, 1.02f)) h_half = __fmul_rn(h_half, 0.90f);
                if (s_t_1024 > __fmul_rn(s_2_1024, 1.02f)) h_2t = __fmul_rn(h_2t, 0.90f);
                const float eps = 1e-6f;
                float r2 = __fdiv_rn(__fadd_rn(s_2_256, eps), __fadd_rn(s_t_256, eps));
                if (r2 < 1.10f) h_2t = __fmul_rn(h_2t, 0.75f);
                if (r2 < 1.00f) h_2t = __fmul_rn(h_2t, 0.75f);
                float rh = __fdiv_rn(__fadd_rn(s_h_1024, eps), __fadd_rn(s_t_1024, eps));
                if (rh < 1.10f) h_half = __fmul_rn(h_half, 0.75f);
                if (rh < 1.00f) h_half = __fmul_rn(h_half, 0.75f);
                float lb[3] = {tb, t2, th}, ls[3] = {h_t, h_2t, h_half};
                int nl = 0;
                for (int q = 0; q < 3; ++q)
                    if (lb[q] >= cfg.min_bpm && lb[q] <= cfg.max_bpm) {
                        float s = ls[q];
                        if (lb[q] > 210.0f) s = __fmul_rn(s, 0.80f);
                        else if (lb[q] > 180.0f) s = __fmul_rn(s, 0.90f);
                        else if (lb[q] < 60.0f) s = __fmul_rn(s, 0.92f);
                        lb[nl] = lb[q];
                        ls[nl] = s;
                        ++nl;
                    }
                if (nl == 0) continue;
                // stable sort desc of <= 3 entries
                for (int a = 1; a < nl; ++a) {
                    float xb = lb[a], xs = ls[a];
                    int j = a;
                    while (j > 0 && ls[j - 1] < xs) { lb[j] = lb[j - 1]; ls[j] = ls[j - 1]; --j; }
                    lb[j] = xb;
                    ls[j] = xs;
                }
                float second = nl > 1 ? ls[1] : 0.0f;
                float margin = __fsub_rn(ls[0], second);
                float ch_b = lb[0], ch_s = ls[0];
                if (fabsf(__fsub_rn(ch_b, tb)) > 1e-3f && margin < cfg.mr_margin) { ch_b = tb; ch_s = h_t; }
                if (margin < cfg.mr_margin && cfg.mr_human_prior && ch_b >= 70.0f && ch_b <= 180.0f && margin < 0.05f) ch_s = __fadd_rn(ch_s, 0.05f);
                hb[nh] = ch_b;
                hs[nh] = ch_s;
                ++nh;
            }
            if (nh > 0) {
                for (int a = 1; a < nh; ++a) {  // stable sort by score desc (:532-536)
                    float xb = hb[a], xs = hs[a];
                    int j = a;
                    while (j > 0 && hs[j - 1] < xs) { hb[j] = hb[j - 1]; hs[j] = hs[j - 1]; --j; }
                    hb[j] = xb;
                    hs[j] = xs;
                }
                float ub[8], us[8];
                int nu = 0;
                for (int a = 0; a < nh && nu < 8; ++a) {
                    bool dup = false;
                    for (int q = 0; q < nu; ++q) dup |= fabsf(__fsub_rn(ub[q], hb[a])) < 0.75f;
                    if (dup) continue;
                    ub[nu] = hb[a];
                    us[nu] = hs[a];
                    ++nu;
                }
                float bb = ub[0], bs = us[0];
                if (bb >= 170.0f) {  // fold-down (:698-724)
                    float half = __fmul_rn(bb, 0.5f);
                    if (half >= 70.0f && half <= 120.0f) {
                        uint32_t ab, ah;
                        float sb_ = total_support(bb, &ab), sh = total_support(half, &ah);
                        float ratio = sb_ > 0.0f ? __fdiv_rn(sh, sb_) : 0.0f;
                        if (ah >= 3 && sh > 0.0f && sb_ > 0.0f && ratio >= 0.45f) { bb = half; bs = sh; }
                    }
                }
                if (bb <= 80.0f) {  // fold-up (:727-751)
                    float dbl = __fmul_rn(bb, 2.0f);
                    if (dbl >= 70.0f && dbl <= 180.0f) {
                        uint32_t ab, ad;
                        float sb_ = total_support(bb, &ab), sd = total_support(dbl, &ad);
                        float ratio = sb_ > 0.0f ? __fdiv_rn(sd, sb_) : 0.0f;
                        if (ad >= 2 && sd > 0.0f && sb_ > 0.0f && ratio >= 0.55f) { bb = dbl; bs = sd; }
                    }
                }
                best_bpm_s = bb;
                best_score_s = bs;
                second_s = nu > 1 ? us[1] : 0.0f;
                mr_ok = 1;
                // triplet family candidates (:764-804)
                if (bb >= 70.0f && bb <= 180.0f && nn > 0) {
                    const float family[5] = {1.0f, 3.0f / 2.0f, 2.0f / 3.0f, 4.0f / 3.0f, 3.0f / 4.0f};
                    int nf = 0;
                    for (int q = 0; q < 5; ++q) {
                        float bpm = __fmul_rn(bb, family[q]);
                        if (!(isfinite(bpm) && bpm >= cfg.min_bpm && bpm <= cfg.max_bpm)) continue;
                        if (!(bpm >= 70.0f && bpm <= 180.0f)) continue;
                        uint32_t ag;
                        float sup = total_support(bpm, &ag);
                        if (ag < 2 || sup <= 0.0f) continue;
                        fam_bpm[nf] = bpm;
                        fam_support[nf] = sup;
                        ++nf;
                    }
                    n_fam = nf;
                    if (nf >= 2) {
                        float bsup = 0.0f;
                        for (int q = 0; q < nf; ++q) bsup = fmaxf(bsup, fam_support[q]);
                        bsup = fmaxf(bsup, 1e-6f);
                        float max_alt = 0.0f;
                        for (int q = 0; q < nf; ++q)
                            if (fabsf(__fsub_rn(fam_bpm[q], bb)) > 0.75f) max_alt = fmaxf(max_alt, __fdiv_rn(fam_support[q], bsup));
                        if (max_alt >= 0.45f) run_family = 1;
                    }
                }
                if (run_family) {  // novelty total (:594), left-to-right
                    float tot = 0.0f;
                    for (uint32_t i = 0; i < nn; ++i) tot = __fadd_rn(tot, nov[i]);
                    s_total = fmaxf(tot, 1e-6f);
                }
            }
        }
    }
    __syncthreads();
    if (!mr_ok) return;
    if (run_family) {
        const int nf = n_fam;
        for (int q = 0; q < nf; ++q) {
            float a = block_beat_contrast(nov, nn, s_total, T.sr, 512, fam_bpm[q], sred);
            if (threadIdx.x == 0) fam_align[q] = a;
        }
        float cur_align = block_beat_contrast(nov, nn, s_total, T.sr, 512, best_bpm_s, sred);
        __syncthreads();
        if (threadIdx.x == 0) {
            float bsup = 0.0f;
            for (int q = 0; q < nf; ++q) bsup = fmaxf(bsup, fam_support[q]);
            bsup = fmaxf(bsup, 1e-6f);
            int ch = 0;
            float ch_score = -1e9f;
            for (int q = 0; q < nf; ++q) {
                float sn = clamp_rs(__fdiv_rn(fam_support[q], bsup), 0.0f, 1.0f);
                float sc = __fadd_rn(fam_align[q], __fmul_rn(0.35f, sn));
                if (sc > ch_score) { ch = q; ch_score = sc; }
            }
            if (fabsf(__fsub_rn(fam_bpm[ch], best_bpm_s)) > 0.75f && fam_align[ch] >= __fadd_rn(cur_align, 0.40f)) {
                best_bpm_s = fam_bpm[ch];
                best_score_s = fam_support[ch];
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const float bb = best_bpm_s, bs = best_score_s;
        float conf = bs > 1e-6f ? clamp_rs(__fdiv_rn(fmaxf(__fsub_rn(bs, second_s), 0.0f), bs), 0.0f, 1.0f) : 0.0f;
        uint32_t agree = 0;
        if (mr_lookup(c256, n256, bb, tol) > 0.0f) ++agree;
        if (mr_lookup(c512, n512, bb, tol) > 0.0f) ++agree;
        if (mr_lookup(c1024, n1024, bb, tol) > 0.0f) ++agree;
        // acceptance rule (lib.rs:515-545)
        const TempoEstDev& base = T.est[cfg.bs];
        float rel = base.bpm > 1e-6f ? fmaxf(__fdiv_rn(bb, base.bpm), __fdiv_rn(base.bpm, bb)) : 1.0f;
        bool fam_rel = fabsf(__fsub_rn(rel, 2.0f)) < 0.05f || fabsf(__fsub_rn(rel, 1.5f)) < 0.05f || fabsf(__fsub_rn(rel, 4.0f / 3.0f)) < 0.05f;
        bool forbid = base.bpm <= 180.0f && bb > 180.0f;
        bool better = !forbid && (conf >= __fadd_rn(base.confidence, 0.05f) || (agree > base.agreement && conf >= __fmul_rn(base.confidence, 0.90f)) ||
                                  ((T.trap_low || T.trap_high) && fam_rel && conf >= __fmul_rn(base.confidence, 0.88f) &&
                                   ((bb >= 70.0f && bb <= 180.0f) || base.bpm > 180.0f)));
        if (better) {
            T.mr_used = 1;
            T.bpm = bb;
            T.bpm_confidence = conf;
            T.chosen_agree = agree;
        }
    }
}

// ---- final BPM selection (lib.rs:814-900, default + force_legacy branches) ------------------------
__global__ void final_bpm_kernel(TrackDev* tr, int n_tracks, DevCfg cfg) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tracks) return;
    TrackDev& T = tr[t];
    if (T.status != 0) return;
    float bpm = 0.0f, conf = 0.0f;
    if (cfg.force_legacy) {
        if (T.legacy.ok) { bpm = T.legacy.bpm; conf = T.legacy.confidence; }
    } else if (T.est[cfg.bs].ok) {
        if (T.perc_used == 1) { bpm = T.perc_bpm; conf = T.perc_conf; }
        else if (T.mr_used == 1) { bpm = T.bpm; conf = T.bpm_confidence; }
        else { bpm = T.est[cfg.bs].bpm; conf = T.est[cfg.bs].confidence; }
    } else if (T.legacy.ok) {
        bpm = T.legacy.bpm;
        conf = T.legacy.confidence;
    }
    if (!cfg.force_legacy && cfg.bpm_fusion) {  // lib.rs:819-892: validator mode — the tempogram BPM is never overridden
        if (T.est[cfg.bs].ok && bpm > 0.0f) {
            const float l_bpm = T.legacy.ok ? T.legacy.bpm : 0.0f;
            const float l_conf = clamp_rs(T.legacy.ok ? T.legacy.confidence : 0.0f, 0.0f, 1.0f);
            float cf = clamp_rs(conf, 0.0f, 1.0f);
            bool agreement = false;
            if (l_bpm > 0.0f) {
                const float d[5] = {fabsf(__fsub_rn(l_bpm, bpm)), fabsf(__fsub_rn(l_bpm, __fmul_rn(bpm, 0.5f))), fabsf(__fsub_rn(l_bpm, __fmul_rn(bpm, 2.0f))),
                                    fabsf(__fsub_rn(l_bpm, __fmul_rn(bpm, 2.0f / 3.0f))), fabsf(__fsub_rn(l_bpm, __fmul_rn(bpm, 3.0f / 2.0f)))};
                for (int q = 0; q < 5; ++q) agreement |= d[q] <= 2.0f;
            }
            if (agreement) cf = clamp_rs(__fadd_rn(cf, __fmul_rn(0.12f, l_conf)), 0.0f, 1.0f);
            else if (l_bpm > 0.0f) cf = clamp_rs(__fmul_rn(cf, 0.90f), 0.0f, 1.0f);
            conf = cf;
        }  // tempogram unavailable: the legacy estimate chosen above stands
    }
    T.bpm = bpm;
    T.bpm_confidence = conf;
}

// ---- percussive tempogram fallback: acceptance rule of lib.rs:621-662, one thread per listed track ------------
__global__ void perc_accept_kernel(TrackDev* tr, const int32_t* __restrict__ list, int n, int bs) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    TrackDev& T = tr[list[i]];
    if (T.status != 0 || !T.est[bs].ok) return;
    T.perc_used = 0;
    const TempoEstDev& pe = T.est[SLOT_PERC];
    if (!pe.ok) return;  // "Percussive tempogram fallback failed"
    const TempoEstDev& base = T.est[bs];
    const float cb = T.mr_used == 1 ? T.bpm : base.bpm;  // chosen_est after the multi-resolution decision
    const float cc = T.mr_used == 1 ? T.bpm_confidence : base.confidence;
    const uint32_t ca = T.chosen_agree;
    const float rel = cb > 1e-6f ? fmaxf(__fdiv_rn(pe.bpm, cb), __fdiv_rn(cb, pe.bpm)) : 1.0f;
    const bool family_related = fabsf(__fsub_rn(rel, 2.0f)) < 0.05f || fabsf(__fsub_rn(rel, 1.5f)) < 0.05f || fabsf(__fsub_rn(rel, 4.0f / 3.0f)) < 0.05f ||
                                fabsf(__fsub_rn(rel, 3.0f / 2.0f)) < 0.05f || fabsf(__fsub_rn(rel, 2.0f / 3.0f)) < 0.05f || fabsf(__fsub_rn(rel, 3.0f / 4.0f)) < 0.05f;
    const bool forbid_promote_high = cb <= 180.0f && pe.bpm > 180.0f;
    const bool base_low_trap = T.trap_low || base.bpm < 95.0f;
    const bool percussive_in_common = pe.bpm >= 70.0f && pe.bpm <= 180.0f;
    const bool p_better = !forbid_promote_high && family_related && percussive_in_common &&
                          (pe.confidence >= __fadd_rn(cc, 0.04f) || (base_low_trap && pe.confidence >= __fmul_rn(cc, 0.85f)) ||
                           (pe.agreement > ca && pe.confidence >= __fmul_rn(cc, 0.92f)));
    if (p_better) {
        T.perc_used = 1;
        T.perc_bpm = pe.bpm;
        T.perc_conf = pe.confidence;
    }
}

void launch_perc_accept(const WaveCtx& c, const int32_t* d_list, int n_list) {
    if (n_list == 0) return;
    perc_accept_kernel<<<(n_list + 127) / 128, 128, 0, c.stream>>>(c.tracks, d_list, n_list, c.cfg.bs);
    count_launch("hpss");
}

// ---- metadata.tempogram_candidates (lib.rs:684-697, 740-752): the candidate list of the chosen estimate ------------
// base list, the hop-512 list re-flagged against the multi-resolution winner (multi_resolution.rs:888-891) or the
// percussive list; `selected` = within 0.75 BPM of the chosen estimate.
__global__ void emit_candidates_kernel(TrackDev* tr, const float* fa, float* oa, int n_tracks, DevCfg cfg) {
    TrackDev& T = tr[blockIdx.x];
    if ((int)blockIdx.x >= n_tracks) return;
    if (threadIdx.x == 0) T.n_cand_out = -1;
    if (T.status != 0 || !T.est[cfg.bs].ok || cfg.force_legacy || !cfg.emit_cands) return;
    int slot = cfg.bs;
    uint32_t n = T.est[cfg.bs].n_cands;
    float best = T.est[cfg.bs].bpm;
    if (T.perc_used == 1) {
        slot = SLOT_PERC;
        n = T.est[SLOT_PERC].n_cands;
        best = T.est[SLOT_PERC].bpm;
    } else if (T.mr_used == 1) {
        slot = 0;  // the hop-512 list of the multi-resolution pass
        n = min(T.est[0].n_cands, max(cfg.mr_top_k, 1u));
        best = T.bpm;  // multi-resolution winner (written by multires_fusion_kernel)
    }
    const TempoCandDev* c = reinterpret_cast<const TempoCandDev*>(fa + T.cands[slot]);
    float* o = oa + T.cand_out;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        o[5 * i + 0] = c[i].bpm;
        o[5 * i + 1] = c[i].score;
        o[5 * i + 2] = c[i].fft_norm;
        o[5 * i + 3] = c[i].ac_norm;
        o[5 * i + 4] = fabsf(__fsub_rn(c[i].bpm, best)) < 0.75f ? 1.0f : 0.0f;
    }
    if (threadIdx.x == 0) T.n_cand_out = (int32_t)n;
}

void launch_emit_candidates(const WaveCtx& c) {
    if (!c.cfg.emit_cands) return;
    emit_candidates_kernel<<<c.n_tracks, 64, 0, c.stream>>>(c.tracks, c.fa, c.oa, c.n_tracks, c.cfg);
    count_launch("tempogram");
}

void launch_tempogram(const WaveCtx& c, int h, const int32_t* d_list, int n_list) {
    if (n_list == 0 || c.max_F[h] < 2) return;
    dim3 g5(MAX_VARIANTS, n_list);
    novelty_kernel<<<g5, 256, 0, c.stream>>>(c.tracks, d_list, c.srtab, c.sr_index, h, c.fa, c.cfg);
    count_launch("tempogram");
    tgfft_kernel<<<g5, 512, 0, c.stream>>>(c.tracks, d_list, c.srtab, c.sr_index, h, c.fa);
    count_launch("tempogram");
    const bool fine = fine_bpm_grid(c.cfg);
    {
        static bool attr_dev[2][64] = {};  // function attributes are per device
        int dev = 0;
        cudaGetDevice(&dev);
        if (!attr_dev[fine][dev & 63]) {
            cudaFuncSetAttribute(fine ? tgac_lag_kernel : tgac_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TGAC_SMEM_FLOATS * sizeof(float));
            attr_dev[fine][dev & 63] = true;
        }
        const uint32_t want = c.max_F[h];  // novelty length upper bound of the wave
        const uint32_t smem_floats = want <= TGAC_SMEM_FLOATS ? want : 0;  // curves that do not fit stay in global memory
        if (fine) tgac_lag_kernel<<<g5, 256, smem_floats * sizeof(float), c.stream>>>(c.tracks, d_list, c.srtab, c.sr_index, h, c.fa, c.cfg, smem_floats);
        else tgac_kernel<<<g5, 256, smem_floats * sizeof(float), c.stream>>>(c.tracks, d_list, c.srtab, c.sr_index, h, c.fa, c.cfg, smem_floats);
    }
    count_launch("tempogram");
    const uint32_t top_n = (h == c.cfg.bs || h == SLOT_PERC) ? c.cfg.base_top_n : c.cfg.mr_aux_k;
    if (fine) score_kernel<true><<<n_list, 256, 0, c.stream>>>(c.tracks, d_list, c.srtab, c.sr_index, h, c.fa, c.cfg, top_n);
    else score_kernel<false><<<n_list, 256, 0, c.stream>>>(c.tracks, d_list, c.srtab, c.sr_index, h, c.fa, c.cfg, top_n);
    count_launch("tempogram");
}

void launch_escalation_gate(const WaveCtx& c) {
    escalation_gate_kernel<<<(c.n_tracks + 127) / 128, 128, 0, c.stream>>>(c.tracks, c.fa, c.n_tracks, c.cfg);
    count_launch("tempogram");
}

void launch_escalation_compact(const WaveCtx& c, int32_t* d_list, int32_t* d_count, uint64_t slot_base, uint64_t slot_stride, uint32_t n_slots) {
    escalation_compact_kernel<<<1, 1024, 0, c.stream>>>(c.tracks, c.n_tracks, d_list, d_count, slot_base, slot_stride, n_slots > 0 ? n_slots : 1u);
    count_launch("tempogram");
}

void launch_multires_fusion(const WaveCtx& c, const int32_t* d_list, int n_list) {
    if (n_list == 0) return;
    multires_fusion_kernel<<<n_list, 128, 0, c.stream>>>(c.tracks, d_list, c.fa, c.cfg);
    count_launch("multires");
}

void launch_final_bpm(const WaveCtx& c) {
    final_bpm_kernel<<<(c.n_tracks + 127) / 128, 128, 0, c.stream>>>(c.tracks, c.n_tracks, c.cfg);
    count_launch("tempogram");
}

}  // namespace sb
