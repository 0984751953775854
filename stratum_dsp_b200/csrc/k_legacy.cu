// Legacy BPM estimator — reference period/mod.rs:216-404 (estimate_bpm_with_guardrails):
//   onset-list autocorrelation via FFT        period/autocorrelation.rs:99-338
//   comb-filterbank scoring of the BPM grid   period/comb_filter.rs:96-215, 342-397
//   candidate merge + boosts + guardrails     period/candidate_filter.rs:51-443, period/mod.rs:242-404
// Always computed (lib.rs:294-329); its estimate is used only when the tempogram produced nothing,
// but its hard errors propagate to the caller.
//
// One CTA per track.  The ACF is IFFT(|FFT(x)|^2)/N on the binary onset signal zero-padded to
// next_pow2(2 len); both transforms are the SFFT DAG over ping-pong buffers in global memory.  The
// comb filterbank is a nearest-neighbour search per (BPM, beat) — not a dense contraction — so one
// thread walks one BPM hypothesis with a moving cursor over the sorted onsets (first-minimum rule of
// `min_by_key` on the truncated distance, comb_filter.rs:371-386).  Grids of more than AC_CAP hypotheses are scored
// beforehand by comb_kernel across CTAs; legacy_kernel then only selects the head of the confidence order.
#include "fft.cuh"
#include "framed.cuh"
#include "kernels.h"

namespace sb {

constexpr int LG_MAX_ACF = 160;   // ACF peak candidates kept
constexpr int LG_MAX_GROUPS = 192;
constexpr int LG_COMB_TOP = 10;   // comb candidates legacy_merge reads (candidate_filter.rs:228-262 keeps the top 10)

struct LgCand {
    float bpm, conf;
};
struct LgEst {
    float bpm, conf;
    uint32_t cnt;
};

__device__ __forceinline__ bool in_range(float b, float lo, float hi) { return b >= lo && b <= hi; }

// merge_bpm_candidates + guardrails + preferred-candidate promotion; thread 0 only.
__device__ inline void legacy_merge(LgCand* ac, int n_ac, const LgCand* comb, int n_comb, LgEst* est, const DevCfg& cfg, TempoEstDev* out) {
    out->ok = 0;
    // preferred ACF candidate is taken before the octave rewrite (period/mod.rs:268-280)
    float pmin = 60.0f, pmax = 180.0f, smin = 0.0f, smax = 0.0f, mp = 0.0f, ms = 0.0f, me = 0.0f;
    if (cfg.legacy_guardrails) {
        pmin = fminf(cfg.lg_pmin, cfg.lg_pmax);
        pmax = fmaxf(cfg.lg_pmin, cfg.lg_pmax);
        smin = fminf(fminf(cfg.lg_smin, cfg.lg_smax), pmin);
        smax = fmaxf(fmaxf(cfg.lg_smin, cfg.lg_smax), pmax);
        mp = isfinite(cfg.lg_mp) ? fmaxf(cfg.lg_mp, 0.0f) : 0.0f;
        ms = isfinite(cfg.lg_ms) ? fmaxf(cfg.lg_ms, 0.0f) : 0.0f;
        me = isfinite(cfg.lg_me) ? fmaxf(cfg.lg_me, 0.0f) : 0.0f;
    }
    bool has_pref = false;
    float pref_bpm = 0.0f;
    for (int i = 0; i < n_ac; ++i)
        if (in_range(ac[i].bpm, pmin, pmax)) {
            has_pref = true;
            pref_bpm = ac[i].bpm;
            break;
        }
    if (n_ac == 0 && n_comb == 0) return;
    const float oct = exp2f(50.0f / 1200.0f);
    const int top3 = min(3, n_comb);
    for (int a = 0; a < n_ac; ++a)
        for (int i = 0; i < top3; ++i) {
            const float ratio = ac[a].bpm / comb[i].bpm;
            if (fabsf(ratio / 2.0f - 1.0f) < (oct - 1.0f)) {
                const bool ok = in_range(comb[i].bpm, 60.0f, 180.0f) || (ac[a].bpm > 200.0f || ac[a].bpm < 30.0f);
                if (ok) {
                    ac[a].bpm = comb[i].bpm;
                    break;
                }
            }
        }
    for (int a = 0; a < n_ac; ++a)
        for (int i = 0; i < top3; ++i) {
            const float ratio = comb[i].bpm / ac[a].bpm;
            if (fabsf(ratio / 2.0f - 1.0f) < (oct - 1.0f)) {
                if (in_range(comb[i].bpm, 60.0f, 180.0f)) {
                    ac[a].bpm = comb[i].bpm;
                    break;
                }
            }
        }
    bool disagree = false;
    if (n_ac > 0 && n_comb > 0) {
        const float d = fabsf(ac[0].bpm - comb[0].bpm);
        disagree = d > 10.0f && d < 50.0f;
    }
    // limited lists (candidate_filter.rs:228-262): top 10 + in-range extras not within 1 BPM of a kept one.
    // `acl` is built in place behind a write cursor: kept entries never move past their source index.
    __shared__ LgCand acl[LG_MAX_ACF];
    int n_acl = min(10, n_ac);
    for (int i = 0; i < n_acl; ++i) acl[i] = ac[i];
    for (int i = 0; i < n_ac; ++i) {
        if (in_range(ac[i].bpm, 60.0f, 180.0f)) {
            bool near = false;
            for (int j = 0; j < n_acl; ++j)
                if (fabsf(acl[j].bpm - ac[i].bpm) < 1.0f) near = true;
            if (!near && n_acl < LG_MAX_ACF) acl[n_acl++] = ac[i];
        }
    }
    const int n_cl = min(10, n_comb);
    // greedy +-2 BPM grouping with running mean (:268-306)
    __shared__ float g_bpm[LG_MAX_GROUPS], g_total[LG_MAX_GROUPS], g_mx[LG_MAX_GROUPS];
    __shared__ uint32_t g_cnt[LG_MAX_GROUPS];
    int ng = 0;
    auto add = [&](const LgCand& c) {
        for (int g = 0; g < ng; ++g)
            if (fabsf(c.bpm - g_bpm[g]) <= 2.0f) {
                g_bpm[g] = (g_bpm[g] * (float)g_cnt[g] + c.bpm) / (float)(g_cnt[g] + 1);
                g_total[g] = g_total[g] + c.conf;
                g_cnt[g] += 1;
                g_mx[g] = fmaxf(g_mx[g], c.conf);
                return;
            }
        if (ng < LG_MAX_GROUPS) {
            g_bpm[ng] = c.bpm;
            g_total[ng] = c.conf;
            g_cnt[ng] = 1;
            g_mx[ng] = c.conf;
            ++ng;
        }
    };
    for (int i = 0; i < n_acl; ++i) add(acl[i]);
    for (int i = 0; i < n_cl; ++i) add(comb[i]);
    for (int g = 0; g < ng; ++g) {
        float conf;
        if (g_cnt[g] >= 2) {
            const float avg = g_total[g] / (float)g_cnt[g];
            conf = fminf((avg + g_mx[g]) / 2.0f * 1.2f, 1.0f);
        } else {
            conf = fminf(g_total[g], 1.0f);
        }
        if (disagree && g_cnt[g] == 1) conf = conf * 0.7f;
        est[g] = LgEst{g_bpm[g], conf, g_cnt[g]};
    }
    // boost_consensus_candidates (:51-112)
    const int a5 = min(5, n_acl), c5 = min(5, n_cl);
    auto harm = [](float x, float y) {
        const float r = fmaxf(x / y, y / x);
        return fabsf(r - 2.0f) < 0.1f || fabsf(r - 1.5f) < 0.1f || fabsf(r - 0.75f) < 0.1f;
    };
    for (int g = 0; g < ng; ++g) {
        bool ad = false, cd = false, ah = false, ch = false;
        for (int i = 0; i < a5; ++i) {
            if (fabsf(acl[i].bpm - est[g].bpm) < 2.5f) ad = true;
            if (harm(acl[i].bpm, est[g].bpm)) ah = true;
        }
        for (int i = 0; i < c5; ++i) {
            if (fabsf(comb[i].bpm - est[g].bpm) < 2.5f) cd = true;
            if (harm(comb[i].bpm, est[g].bpm)) ch = true;
        }
        if (ad && cd) est[g].conf = est[g].conf * 1.5f;
        else if ((ad && ch) || (cd && ah)) est[g].conf = est[g].conf * 1.3f;
        if (cd && in_range(est[g].bpm, 60.0f, 180.0f)) est[g].conf = est[g].conf * 1.4f;
    }
    bool reasonable_top5 = false;
    for (int g = 0; g < min(5, ng); ++g)
        if (in_range(est[g].bpm, 60.0f, 180.0f)) reasonable_top5 = true;
    if (!reasonable_top5)
        for (int g = 0; g < ng; ++g)
            if (in_range(est[g].bpm, 60.0f, 180.0f)) {
                est[g].conf = est[g].conf * 2.0f;
                break;
            }
    // final ordering (:385-433).  The comparator is not a strict weak order; the documented semantics
    // (DESIGN.md, oracle/so_legacy.cpp) are those of a stable insertion sort over it.
    auto cmp3 = [](const LgEst& a, const LgEst& b) -> int {
        const bool ai = in_range(a.bpm, 60.0f, 180.0f), bi = in_range(b.bpm, 60.0f, 180.0f);
        const float ae = ai ? a.conf : a.conf * 0.5f, be = bi ? b.conf : b.conf * 0.5f;
        const int ec = (be < ae) ? -1 : ((be > ae) ? 1 : 0);
        if (fabsf(ae - be) < 0.5f) {
            if (ai && !bi) return -1;
            if (!ai && bi) return 1;
        }
        if (ec != 0) return ec;
        return (b.cnt < a.cnt) ? -1 : ((b.cnt > a.cnt) ? 1 : 0);
    };
    for (int i = 1; i < ng; ++i) {
        const LgEst x = est[i];
        int j = i;
        while (j > 0 && cmp3(x, est[j - 1]) < 0) {
            est[j] = est[j - 1];
            --j;
        }
        est[j] = x;
    }
    if (cfg.legacy_guardrails) {  // period/mod.rs:296-321
        for (int g = 0; g < ng; ++g) {
            float mul;
            const float b = est[g].bpm;
            if (!isfinite(b)) mul = 0.0f;
            else if (in_range(b, pmin, pmax)) mul = mp;
            else if (in_range(b, smin, smax)) mul = ms;
            else mul = me;
            est[g].conf = est[g].conf * mul;
        }
        for (int i = 1; i < ng; ++i) {  // stable sort by confidence desc
            const LgEst x = est[i];
            int j = i;
            while (j > 0 && est[j - 1].conf < x.conf) {
                est[j] = est[j - 1];
                --j;
            }
            est[j] = x;
        }
    }
    int first = 0;
    if (has_pref)
        for (int g = 0; g < ng; ++g)
            if (fabsf(est[g].bpm - pref_bpm) < 2.0f) {
                first = g;  // moved to the front (period/mod.rs:323-334); only element 0 is consumed
                break;
            }
    if (ng > 0) {
        out->bpm = est[first].bpm;
        out->confidence = est[first].conf;
        out->agreement = est[first].cnt;
        out->ok = 1;
    }
}

// score_bpm_candidate (comb_filter.rs:342-397): share of the expected beats k * period that have an onset within tol * period.  The
// nearest onset is found with a cursor moving over the sorted onsets (first minimum of `min_by_key` on the truncated distance, :371-386).
__device__ inline float comb_score(const int32_t* on, uint32_t n_on, uint32_t sr, float bpm) {
    const float tol = clamp_rs(0.1f * (120.0f / bpm), 0.05f, 0.15f);
    const float period = (60.0f * (float)sr) / bpm;
    float score = 0.0f;
    if (period >= 1.0f) {  // `period < 1` is a NumericalError in the reference; unreachable for sr >= 240 / 60
        const float tol_s = period * tol;
        const float last = (float)on[n_on - 1];
        const uint32_t num_beats = as_u32(ceilf(last / period)) + 1;
        uint32_t aligned = 0, cur = 0;
        for (uint32_t k = 0; k < num_beats; ++k) {
            const float eb = (float)k * period;
            while (cur + 1 < n_on && (float)on[cur + 1] <= eb) ++cur;
            const uint32_t lo = cur >= 3 ? cur - 3 : 0, hi = min(cur + 4, n_on);
            uint32_t best_i = lo;
            uint64_t best_k = ~0ull;
            for (uint32_t i = lo; i < hi; ++i) {
                const uint64_t key = as_u64(fabsf((float)on[i] - eb));
                if (key < best_k) {
                    best_k = key;
                    best_i = i;
                }
            }
            const float d = fabsf((float)on[best_i] - eb);
            if (d <= tol_s) ++aligned;
        }
        score = num_beats > 0 ? (float)aligned / (float)num_beats : 0.0f;
    }
    return score;
}

// ---- comb filterbank of a fine BPM grid: one thread per hypothesis, one CTA per (256 hypotheses, track) -------------------------
// A 60-minute mix at 0.01 BPM is about 20 000 hypotheses x 7 000 beats: spread over CTAs instead of one per track.
__global__ void __launch_bounds__(256) comb_kernel(const TrackDev* tr, float* fa, const int32_t* __restrict__ ia, DevCfg cfg) {
    const TrackDev& T = tr[blockIdx.y];
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (T.status != 0 || T.n_on_final < 2 || b >= cfg.n_comb) return;
    fa[T.lg_comb + b] = comb_score(ia + T.on_final, T.n_on_final, T.sr, cfg.bpm_tab[b]);
}

template <bool FINE>  // FINE: more than AC_CAP hypotheses, scored beforehand by comb_kernel
__global__ void __launch_bounds__(256) legacy_kernel(TrackDev* tr, float* fa, const int32_t* __restrict__ ia, DevCfg cfg) {
    __shared__ float sred[32];
    __shared__ float top_val[8];
    __shared__ int top_w[8], top_idx[LG_COMB_TOP];
    __shared__ LgCand ac[LG_MAX_ACF];
    __shared__ LgCand comb[AC_CAP];
    __shared__ float craw[AC_CAP], cbpm[AC_CAP];
    __shared__ LgEst est[LG_MAX_GROUPS];
    __shared__ int s_nac, s_ncomb;
    TrackDev& T = tr[blockIdx.x];
    if (threadIdx.x == 0) T.legacy.ok = 0;
    if (T.status != 0) return;
    const uint32_t n_on = T.n_on_final;
    if (n_on < 2) return;  // lib.rs:299-307: legacy skipped
    const int32_t* on = ia + T.on_final;
    const uint32_t hop = cfg.hop;  // lib.rs:310: config.hop_size
    const uint32_t sr = T.sr;
    // ---- autocorrelation candidates ----
    const uint32_t max_frame = (uint32_t)on[n_on - 1] / hop;
    const uint32_t len = max_frame + 1;
    if (len < 2) {
        if (threadIdx.x == 0) {
            T.status = STRATUM_PROCESSING_ERROR;
            T.err_code = 4;  // "Signal too short for autocorrelation"
        }
        return;
    }
    const uint32_t N = next_pow2_u32(2 * len);
    if (threadIdx.x == 0) s_nac = 0;
    float max_acf = 0.0f;
    const float* acf = nullptr;
    if (N <= T.lg_fft) {
        float2* A = reinterpret_cast<float2*>(fa + T.lg_work);
        float2* B = A + T.lg_fft;
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) A[i] = make_float2(0.0f, 0.0f);
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n_on; i += blockDim.x) {
            const uint32_t f = (uint32_t)on[i] / hop;
            if (f < len) A[f].x = 1.0f;  // duplicates write the same value
        }
        __syncthreads();
        const uint32_t tws = T.lg_fft / N;
        float2* Z = cta_cfft(A, B, T.lg_tw, N, tws);
        float2* O = (Z == A) ? B : A;
        for (uint32_t i = threadIdx.x; i < N; i += blockDim.x) {  // x *= conj(x), then conjugate for the inverse
            const float2 v = Z[i];
            const float re = v.x * v.x - v.y * (-v.y);
            const float im = v.x * (-v.y) + v.y * v.x;
            Z[i] = make_float2(re, -im);
        }
        __syncthreads();
        float2* R = cta_cfft(Z, O, T.lg_tw, N, tws);
        const float scale = 1.0f / (float)N;
        float* out = reinterpret_cast<float*>(R == A ? B : A);  // the other buffer is free now
        for (uint32_t i = threadIdx.x; i < len; i += blockDim.x) {
            const float v = fmaxf(R[i].x * scale, 0.0f);
            out[i] = v;
            max_acf = fmaxf(max_acf, v);
        }
        max_acf = block_max(max_acf, sred);
        __syncthreads();
        acf = out;
    }
    const uint32_t lag_min = as_u32(ceilf((60.0f * (float)sr) / (cfg.max_bpm * (float)hop)));
    const uint32_t lag_max = as_u32(floorf((60.0f * (float)sr) / (cfg.min_bpm * (float)hop)));
    if (acf && !(lag_min >= lag_max || lag_min >= len || lag_max >= len)) {
        const float* a = acf + lag_min;
        const uint32_t L = lag_max - lag_min + 1;
        float mx = 0.0f;
        for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) mx = fmaxf(mx, a[i]);
        mx = block_max(mx, sred);
        if (threadIdx.x == 0 && !(mx < 1e-10f)) {  // find_peaks_in_acf (:282-338)
            const float min_prom = mx * 0.1f;
            __shared__ uint32_t pk_lag[LG_MAX_ACF];
            __shared__ float pk_val[LG_MAX_ACF];
            int np = 0;
            for (uint32_t i = 1; i + 1 < L; ++i) {
                const float v = a[i];
                if (v > a[i - 1] && v > a[i + 1]) {
                    const float prom = v - fmaxf(a[i - 1], a[i + 1]);
                    if (prom >= min_prom) {
                        const uint32_t lag = i + lag_min;
                        if (np == 0 || abs((int)lag - (int)pk_lag[np - 1]) >= 2) {
                            if (np < LG_MAX_ACF) {
                                pk_lag[np] = lag;
                                pk_val[np] = v;
                                ++np;
                            }
                        } else if (v > pk_val[np - 1]) {
                            pk_lag[np - 1] = lag;
                            pk_val[np - 1] = v;
                        }
                    }
                }
            }
            // stable sort by value desc, then bpm/conf, filter, stable sort by confidence desc
            for (int i = 1; i < np; ++i) {
                const float v = pk_val[i];
                const uint32_t l = pk_lag[i];
                int j = i;
                while (j > 0 && pk_val[j - 1] < v) {
                    pk_val[j] = pk_val[j - 1];
                    pk_lag[j] = pk_lag[j - 1];
                    --j;
                }
                pk_val[j] = v;
                pk_lag[j] = l;
            }
            int na = 0;
            for (int i = 0; i < np; ++i) {
                const float bpm = (60.0f * (float)sr) / ((float)pk_lag[i] * (float)hop);
                if (bpm >= cfg.min_bpm && bpm <= cfg.max_bpm) {
                    const float conf = max_acf > 1e-10f ? fminf(pk_val[i] / max_acf, 1.0f) : 0.0f;
                    ac[na++] = LgCand{bpm, conf};
                }
            }
            for (int i = 1; i < na; ++i) {
                const LgCand x = ac[i];
                int j = i;
                while (j > 0 && ac[j - 1].conf < x.conf) {
                    ac[j] = ac[j - 1];
                    --j;
                }
                ac[j] = x;
            }
            s_nac = na;
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) s_ncomb = 0;
    __syncthreads();
    float* raw = fa + T.lg_comb;  // raw scores in hypothesis order
    if constexpr (!FINE) {
        // ---- comb filterbank: one thread per BPM hypothesis ----
        int nb = 0;
        {
            float b = cfg.min_bpm;
            while (b <= cfg.max_bpm + 1e-10f && nb < AC_CAP) {
                ++nb;
                b = b + cfg.bpm_resolution;
            }
        }
        float my_max = 0.0f;
        for (int bi = threadIdx.x; bi < nb; bi += blockDim.x) {
            float bpm = cfg.min_bpm;
            for (int q = 0; q < bi; ++q) bpm = bpm + cfg.bpm_resolution;
            const float score = comb_score(on, n_on, sr, bpm);
            craw[bi] = score;
            cbpm[bi] = bpm;
            raw[bi] = score;
            my_max = fmaxf(my_max, score);
        }
        const float max_score = block_max(my_max, sred);
        __syncthreads();
        for (int bi = threadIdx.x; bi < nb; bi += blockDim.x) craw[bi] = max_score > 1e-10f ? craw[bi] / max_score : 0.0f;
        __syncthreads();
        // stable sort by confidence desc (rank counting), entries below 0.1 dropped (they sort last)
        for (int bi = threadIdx.x; bi < nb; bi += blockDim.x) {
            const float x = craw[bi];
            int r = 0;
            for (int j = 0; j < nb; ++j) r += (craw[j] > x) || (craw[j] == x && j < bi);
            comb[r] = LgCand{cbpm[bi], x};
            if (x >= 0.1f) atomicAdd(&s_ncomb, 1);
        }
    } else {
        // ---- fine grid: comb_kernel wrote the raw scores.  legacy_merge reads the first 10 entries of the confidence order and the
        // count of entries >= 0.1, so the order is only needed that far: top 10 by (confidence desc, index asc) = the stable sort's
        // head.  Selected on the normalised values, as the sort is (the division can tie different raw scores).
        const int nb = (int)cfg.n_comb;
        float my_max = 0.0f;
        for (int bi = threadIdx.x; bi < nb; bi += blockDim.x) my_max = fmaxf(my_max, raw[bi]);
        const float max_score = block_max(my_max, sred);
        auto conf = [&](int bi) { return max_score > 1e-10f ? raw[bi] / max_score : 0.0f; };
        int n_keep = 0;
        for (int bi = threadIdx.x; bi < nb; bi += blockDim.x) n_keep += conf(bi) >= 0.1f;
        if (n_keep) atomicAdd(&s_ncomb, n_keep);
        const int k = block_topk<LG_COMB_TOP>(conf, 0, nb - 1, top_idx, top_val, top_w);
        if ((int)threadIdx.x < k) comb[threadIdx.x] = LgCand{cfg.bpm_tab[top_idx[threadIdx.x]], conf(top_idx[threadIdx.x])};
    }
    __syncthreads();
    if (threadIdx.x == 0) legacy_merge(ac, s_nac, comb, s_ncomb, est, cfg, &T.legacy);
}

void launch_legacy_bpm(const WaveCtx& c) {
    if (fine_bpm_grid(c.cfg)) {
        comb_kernel<<<dim3((c.cfg.n_comb + 255) / 256, c.n_tracks), 256, 0, c.stream>>>(c.tracks, c.fa, c.ia, c.cfg);
        count_launch("legacy_bpm");
        legacy_kernel<true><<<c.n_tracks, 256, 0, c.stream>>>(c.tracks, c.fa, c.ia, c.cfg);
    } else {
        legacy_kernel<false><<<c.n_tracks, 256, 0, c.stream>>>(c.tracks, c.fa, c.ia, c.cfg);
    }
    count_launch("legacy_bpm");
}

}  // namespace sb
