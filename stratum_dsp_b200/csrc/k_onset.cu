// Onset detection kernels: energy flux (reference onset/energy_flux.rs:67-243), per-frame and
// per-frame-pair spectrogram reductions shared by the spectral-flux / HFC detectors
// (onset/spectral_flux.rs:120-157, onset/hfc.rs:132-154) and by the tempogram novelty curves
// (period/novelty.rs:336-836), exact percentile thresholds + peak picking, and the consensus vote
// (onset/consensus.rs:111-287 with the caller-side policy of lib.rs:258-286).
//
// Every sum that feeds a comparison is accumulated in the reference's order (bin 0 upward, one
// rounded multiply and one rounded add per term), one thread per frame / frame pair.
#include <algorithm>

#include "framed.cuh"
#include "kernels.h"

namespace sb {

// frame-region layout (q * fmax + t): 0 rowmax, 1 E, 2 H, 3..5 E_low/mid/high, 6..8 H_low/mid/high
constexpr int FQ_ROWMAX = 0, FQ_E = 1, FQ_H = 2, FQ_EB = 3, FQ_HB = 6;
// pair-region layout: 0 onset spectral flux, 1 SF_full, 2..4 SF_low/mid/high, 5 SF_mel
constexpr int PQ_SFLUX = 0, PQ_SF = 1, PQ_SFB = 2, PQ_MEL = 5;
constexpr int MEL_MAX = 40;

// ---- energy flux onsets ------------------------------------------------------------------------
constexpr int ERMS_SEG = 32;  // hop-blocks per segment of the streamed frame-RMS (framed.cuh)
// hop_size other than 512: the tile form (one lane per frame, any hop), same per-frame sums in the same order
template <int FRAME>
__global__ void __launch_bounds__(128) energy_rms_any_kernel(const float* __restrict__ x, const TrackDev* tr, float* fa, uint32_t hop, int bs) {
    __shared__ float tiles[4][32][33];
    const TrackDev& T = tr[blockIdx.y];
    const uint32_t nf = T.F[bs];
    const uint32_t f0 = (blockIdx.x * 4 + (threadIdx.x >> 5)) * 32;
    if (f0 >= nf || T.status != 0) return;
    framed_rms_warp<FRAME>(x + T.off + T.trim_start, T.m, T.gain, hop, f0, nf, tiles[threadIdx.x >> 5], fa + T.erms);
}

// hop 512: FRAME / 512 lanes per segment (4 at 2048, 8 at 4096, 16 at 8192), ERMS_GPW segments per warp
template <int FRAME>
constexpr int ERMS_GPW = 32 / (FRAME / 512);
template <int FRAME>
__global__ void __launch_bounds__(128) energy_rms_kernel(const float* __restrict__ x, const TrackDev* tr, float* fa) {
    constexpr int GPW = ERMS_GPW<FRAME>;
    __shared__ float tiles[4][2][GPW][33];
    const TrackDev& T = tr[blockIdx.y];
    const uint32_t nf = T.F[0];  // > 0 only when the trimmed track holds a full frame
    const uint32_t seg_first = (blockIdx.x * 4 + (threadIdx.x >> 5)) * GPW;
    if (seg_first * ERMS_SEG >= nf || T.status != 0) return;
    framed_rms_stream_warp<FRAME, 512, ERMS_SEG>(x + T.off + T.trim_start, T.m, T.gain, nf, seg_first, tiles[threadIdx.x >> 5], fa + T.erms);
}

// Shared peak rule of the three detectors (energy_flux.rs:176-217, spectral_flux.rs:183-210, hfc.rs:180-204).
__device__ __forceinline__ bool is_peak(const float* f, uint32_t i, uint32_t L, float thr) {
    if (L < 2) return false;
    float v = f[i];
    if (!(v > thr)) return false;
    if (i == 0) return v >= f[1];
    if (i == L - 1) return v > f[L - 2];
    return v > f[i - 1] && v >= f[i + 1];
}

// Ordered compaction of peak indices of f[0..L) into out (as (i+1)*hop sample positions < m).
__device__ inline uint32_t compact_peaks(const float* f, uint32_t L, float thr, uint32_t hop, uint64_t m, int32_t* out, uint32_t* sc) {
    const uint32_t per = (L + blockDim.x - 1) / blockDim.x;
    const uint32_t a = threadIdx.x * per, b = min(a + per, L);
    uint32_t cnt = 0;
    for (uint32_t i = a; i < b; ++i)
        if (is_peak(f, i, L, thr) && (uint64_t)(i + 1) * hop < m) ++cnt;
    uint32_t total;
    uint32_t pos = block_exclusive_scan(cnt, &total, sc);
    for (uint32_t i = a; i < b; ++i)
        if (is_peak(f, i, L, thr) && (uint64_t)(i + 1) * hop < m) out[pos++] = (int32_t)((i + 1) * hop);
    return total;
}

__global__ void __launch_bounds__(256) energy_onset_kernel(TrackDev* tr, float* fa, int32_t* ia, DevCfg cfg) {
    __shared__ uint32_t sc[34];
    __shared__ float smax[32];
    TrackDev& T = tr[blockIdx.x];
    if (T.status != 0) return;
    const uint32_t nf = T.F[cfg.bs];
    if (threadIdx.x == 0) {
        T.n_on_energy = 0;
        T.onset_method_consensus = 0.0f;
    }
    if (nf < 2) return;
    const uint32_t L = nf - 1;
    const float* rms = fa + T.erms;
    float* flux = fa + T.scratch;
    float mx = 0.0f;
    for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) {
        float v = fmaxf(__fsub_rn(rms[i + 1], rms[i]), 0.0f);
        flux[i] = v;
        mx = fmaxf(mx, v);
    }
    mx = block_max(mx, smax);
    __syncthreads();
    if (mx <= 1e-10f) return;
    const float thr = __fmul_rn(mx, cfg.energy_thr_mul);
    int32_t* out = ia + T.on_energy;
    uint32_t total = compact_peaks(flux, L, thr, cfg.hop, T.m, out, sc);
    __syncthreads();
    if (threadIdx.x == 0) {  // dedupe within hop/2 (energy_flux.rs:224-238)
        uint32_t w = 0;
        for (uint32_t i = 0; i < total; ++i)
            if (w == 0 || out[i] >= out[w - 1] + (int32_t)(cfg.hop / 2)) out[w++] = out[i];
        T.n_on_energy = w;
        T.onset_method_consensus = w > 0 ? 1.0f : 0.0f;
    }
}

// ---- spectrogram reductions --------------------------------------------------------------------
// Two kernels per hop, split by what the consumer needs:
//   seq_feat_kernel — the sums whose value decides a discrete outcome (onset spectral flux, HFC, frame
//     energy): one lane per frame walks the bins in the reference's order; a warp transposes 33x32
//     tiles through shared memory so global loads stay coalesced.  The row maximum it divides by is
//     order-free and comes from the STFT epilogue.
//   par_feat_kernel — everything behind ln(1+x) (SuperFlux full + 3 bands, mel SuperFlux) and the band
//     energies / HFCs, which only reach the BPM through tolerance-level novelty curves: one warp walks a
//     run of 32 consecutive frames, lanes stride the bins (coalesced), ln(1+x) is evaluated once per
//     (frame, bin) and kept in shared memory for the next frame's max filter; reductions are warp trees.
//     Mel bands are folded by one lane per band in ascending-bin order (the reference's order).
// Rows of slot h's spectrogram and their maxima.  The multi-resolution slots share frames with the hop-512 slot (k_stft.cu:
// launch_stft_hop): frame f of the hop-1024 sequence is hop-512 frame 2f, an even frame f of the hop-256 sequence is hop-512 frame f/2,
// bit for bit — only the odd hop-256 frames have rows (and maxima) of their own.  MODE: 0 = the slot's own rows (hop 512, percussive
// component), 1 = hop 256, 2 = hop 1024; a template parameter, with the base pointers hoisted by the caller — a run-time slot test in
// the row loops cost the feature kernels 20 %.
struct SpecRows {
    const float* own;   // the slot's spectrogram
    const float* base;  // the hop-512 spectrogram
    const float* own_max;
    const float* base_max;
};
__device__ __forceinline__ SpecRows spec_rows(const TrackDev& T, const float* fa, int h) {
    return SpecRows{fa + T.hop[h].spec, fa + T.hop[0].spec, fa + T.hop[h].frame + (uint64_t)FQ_ROWMAX * T.hop[h].fmax,
                    fa + T.hop[0].frame + (uint64_t)FQ_ROWMAX * T.hop[0].fmax};
}
template <int MODE, int NB>
__device__ __forceinline__ const float* spec_row(const SpecRows& R, uint32_t f) {
    if (MODE == 1) return (f & 1u) ? R.own + (uint64_t)f * NB : R.base + (uint64_t)(f >> 1) * NB;
    if (MODE == 2) return R.base + (uint64_t)(2 * f) * NB;
    return R.own + (uint64_t)f * NB;
}
template <int MODE>
__device__ __forceinline__ float spec_rowmax(const SpecRows& R, uint32_t f) {
    if (MODE == 1) return (f & 1u) ? R.own_max[f] : R.base_max[f >> 1];
    if (MODE == 2) return R.base_max[2 * f];
    return R.own_max[f];
}

constexpr int FEAT_RUN = 32;
constexpr int HALO = 8;  // superflux radius upper bound (the ABI rejects larger values)

// NB: bins per row (frame_size / 2 + 1)
template <int MODE, int NB>
__global__ void __launch_bounds__(128) seq_feat_kernel(const TrackDev* tr, const int32_t* __restrict__ list, int h, float* fa) {
    // A warp owns 32 consecutive frames f0 .. f0+31 and produces the flux of the 31 pairs inside them: the normalised value
    // x[f][k] / max[f] that frame f contributes as "current" is the same number frame f+1 needs as "previous", so every lane
    // divides once and hands its quotient to the next lane by shuffle (bit-identical to dividing again, half the IEEE
    // divisions).  Consecutive warps overlap by one frame (31 new frames per warp); the duplicated frame's E / H are the
    // same values written twice.
    __shared__ float tiles[4][32][33];
    const int t = list ? list[blockIdx.y] : blockIdx.y;
    const TrackDev& T = tr[t];
    const uint32_t F = T.F[h];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t f0 = (blockIdx.x * 4 + w) * 31;
    if (f0 >= F || T.status != 0) return;
    float(*tile)[33] = tiles[w];
    const HopLayout& HL = T.hop[h];
    float* fr = fa + HL.frame;
    const uint64_t fm = HL.fmax;
    const uint32_t f = f0 + lane;
    const bool valid = f < F;
    const SpecRows R = spec_rows(T, fa, h);
    const float maxc = valid ? spec_rowmax<MODE>(R, f) : 0.0f;
    const bool nc = maxc > 1e-10f;
    // x / max with the frame-constant divisor's correctly rounded reciprocal and one Markstein correction (common.cuh): three
    // instructions per bin instead of the generic division's ten.  x <= max, so the quotient is in [0, 1]; the result is the IEEE
    // quotient unless x < 2^-60 * max, and such a bin's flux term (difference squared) is zero either way.  A row maximum with an
    // all-ones significand or outside [2^-60, 2^60] keeps the generic division.
    const float rmax = nc ? __frcp_rn(maxc) : 0.0f;
    const bool fastdiv = nc && maxc >= 8.6736174e-19f && maxc <= 1.1529215e18f && (__float_as_uint(maxc) & 0x7fffffu) != 0x7fffffu;
    float sflux = 0.0f, E = 0.0f, H = 0.0f;
    auto step = [&](uint32_t k, float cur) {
        const float xc = fastdiv ? div_by_rcp_rn(cur, maxc, rmax) : (nc ? __fdiv_rn(cur, maxc) : 0.0f);   // spectral_flux.rs:120-157
        const float xp = __shfl_up_sync(0xffffffffu, xc, 1);  // the previous frame's normalised bin (lane 0: unused)
        const float d0 = fmaxf(__fsub_rn(xc, xp), 0.0f);
        sflux = __fadd_rn(sflux, __fmul_rn(d0, d0));
        E = __fadd_rn(E, __fmul_rn(cur, cur));
        H = __fadd_rn(H, __fmul_rn(__fmul_rn((float)k, cur), cur));  // hfc.rs:137
    };
    for (uint32_t jb = 0; jb < (NB - 1) / 32; ++jb) {
#pragma unroll 4
        for (int r = 0; r < 32; ++r) {
            const uint32_t fr_ = f0 + r;
            tile[r][lane] = fr_ < F ? spec_row<MODE, NB>(R, fr_)[jb * 32 + lane] : 0.0f;
        }
        __syncwarp();
#pragma unroll 4
        for (int j = 0; j < 32; ++j) step(jb * 32 + j, tile[lane][j]);
        __syncwarp();
    }
    step(NB - 1, valid ? spec_row<MODE, NB>(R, f)[NB - 1] : 0.0f);  // all lanes: the shuffle inside is warp-wide
    if (valid) {
        fr[FQ_E * fm + f] = E;
        fr[FQ_H * fm + f] = H;
        if (lane >= 1) fa[HL.pair + PQ_SFLUX * fm + f - 1] = __fadd_rn(sqrtf(sflux), 0.0f);
    }
}

template <int NB>
struct ParSmem {
    float L[2][NB + 2 * HALO + 7];
    float mel[2][MEL_MAX];
    float part[64];  // partial sums of the mel fold's chunks
};
// Warps per CTA: 4 at 1025 bins (static shared memory, 35 KB); 4 at 2049 (66 KB) and 2 at 4097 (66 KB) in dynamic shared memory,
// so that three CTAs fit an SM at every size.
template <int NB>
constexpr int PAR_WARPS = NB <= 2049 ? 4 : 2;

// K4: the SuperFlux radius is the default 4 (config.rs:634) — the pair pass then gives every lane four CONSECUTIVE bins: the twelve
// previous-frame values their windows cover come from three 16-byte shared loads and the four 9-tap maxima share the maximum of the
// six values common to all windows (17 FMNMX for four bins instead of 36 loads + 36 FMNMX, and a quarter of the shared-memory
// instructions: ncu had the L1/shared pipe at 73 % on the lane-strided version).  Sums are warp trees either way (tolerance-level
// consumers), so only their association changes.
template <bool K4, int MODE, int NB>
__global__ void __launch_bounds__(32 * PAR_WARPS<NB>) par_feat_kernel(const TrackDev* tr, const int32_t* __restrict__ list, const SrTables* srtab,
                                                                     const int32_t* sr_index, int h, float* fa, DevCfg cfg) {
    constexpr int W = PAR_WARPS<NB>;
    ParSmem<NB>* sm;
    if constexpr (NB == 1025) {
        __shared__ __align__(16) ParSmem<NB> sm_static[W];
        sm = sm_static;
    } else {
        extern __shared__ __align__(16) unsigned char par_dyn[];
        sm = reinterpret_cast<ParSmem<NB>*>(par_dyn);
    }
    const int t = list ? list[blockIdx.y] : blockIdx.y;
    const TrackDev& T = tr[t];
    const uint32_t F = T.F[h];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t f0 = (blockIdx.x * W + w) * FEAT_RUN;
    if (f0 >= F || T.status != 0) return;
    ParSmem<NB>& S = sm[w];
    const SrTables& st = srtab[sr_index[t]];
    const HopLayout& HL = T.hop[h];
    float* fr = fa + HL.frame;
    float* pr = fa + HL.pair;
    const uint64_t fm = HL.fmax;
    const SpecRows R = spec_rows(T, fa, h);
    const int K = K4 ? 4 : (int)min(max(cfg.sf_k, 1u), (uint32_t)HALO);
    const int MK = (int)max(cfg.mel_k, 1u);
    const int nm = (int)st.n_mels;
    const int e0 = (int)st.b0, e1 = (int)st.b_low, e2 = (int)st.b_mid, e3 = (int)st.b_hi;
    for (int i = lane; i < NB + 2 * HALO + 7; i += 32) S.L[0][i] = S.L[1][i] = 0.0f;  // halos stay zero: ln(1+x) >= 0 and the reference's running max starts at 0
    __syncwarp();
    int cur = 0;
    const uint32_t f_first = f0 > 0 ? f0 - 1 : 0;
    const uint32_t f_last = min(f0 + FEAT_RUN, F);
    for (uint32_t f = f_first; f < f_last; ++f, cur ^= 1) {
        float* Lc = S.L[cur] + HALO;
        const float* Lp = S.L[cur ^ 1] + HALO;
        const float* row = spec_row<MODE, NB>(R, f);
        const bool emit = f >= f0;           // this warp owns the outputs of frame f
        const bool pair = emit && f >= 1;    // pair (f-1, f) -> index f-1
        // per-band accumulators are selected with predicates, never indexed: a run-time index would put the arrays in local
        // memory and chain every iteration through a store -> load round trip (27 % of the kernel's stall samples in ncu)
        float Eb[3] = {0.0f, 0.0f, 0.0f}, Hb[3] = {0.0f, 0.0f, 0.0f};
        // the row is fetched four 32-bin slices ahead (read-only path: the loads may pass the shared-memory stores of the slices in
        // front of them): ncu had this loop waiting on one global load per slice (long-scoreboard 7.1 warps per issue, issue 47 %).
        // Measured and rejected (round 2, r02s): walking the row band by band with one unpredicated accumulator pair per band, or slice
        // by slice with test-free code for slices inside one band — 25-35 % fewer instructions in this loop, 9-22 % SLOWER: the warp is
        // bound by the dependent chain of the logarithm at 6 warps per scheduler, and the four interleaved slices of this form are what
        // gives it instruction-level parallelism.
        {
            constexpr int PF = 8;  // slices in flight (8 measured 4 % faster than 4: r02H)
            float xq[PF];
#pragma unroll
            for (int u = 0; u < PF; ++u) xq[u] = __ldg(row + 32 * u + lane);
#pragma unroll PF
            for (int b0 = 0; b0 < NB; b0 += 32) {
                const int b = b0 + lane;
                const bool in = b < NB;
                const int u = (b0 >> 5) & (PF - 1);
                const float x = in ? xq[u] : 0.0f;
                if (b + 32 * PF < NB) xq[u] = __ldg(row + b + 32 * PF);
                if (in) Lc[b] = logf(1.0f + fmaxf(x, 0.0f));  // novelty.rs:354
                if (emit && in && b >= e0 && b < e3) {
                    const float xx = x * x, kx = (float)b * x * x;
                    const bool q0 = b < e1, q1 = !q0 && b < e2, q2 = !q0 && !q1;
                    Eb[0] += q0 ? xx : 0.0f;
                    Hb[0] += q0 ? kx : 0.0f;
                    Eb[1] += q1 ? xx : 0.0f;
                    Hb[1] += q1 ? kx : 0.0f;
                    Eb[2] += q2 ? xx : 0.0f;
                    Hb[2] += q2 ? kx : 0.0f;
                }
            }
        }
        __syncwarp();
        float sf = 0.0f, sfb[3] = {0.0f, 0.0f, 0.0f};
        // one bin of the pair pass: pm = max of the previous frame's 2K+1 window around b (novelty.rs:360-420), lc = this frame's value
        auto pair_bin = [&](int b, float pm, float lc) {
            const float d = fmaxf(lc - pm, 0.0f);
            sf += d * d;
            if (b >= e0 && b < e3) {
                const int band = b < e1 ? 0 : (b < e2 ? 1 : 2);
                const int lo = band == 0 ? e0 : (band == 1 ? e1 : e2), hi = band == 0 ? e1 : (band == 1 ? e2 : e3);
                float pmb = pm;
                if (b - K < lo || b + K >= hi) {  // window clipped to the band (novelty.rs:432-441)
                    pmb = 0.0f;
                    for (int j = max(b - K, lo); j < min(b + K + 1, hi); ++j) pmb = fmaxf(pmb, Lp[j]);
                }
                const float db = fmaxf(lc - pmb, 0.0f), dd = db * db;
                sfb[0] += band == 0 ? dd : 0.0f;
                sfb[1] += band == 1 ? dd : 0.0f;
                sfb[2] += band == 2 ? dd : 0.0f;
            }
        };
        if (pair) {
            if (K4) {
#pragma unroll 2
                for (int g = 0; g < (NB - 1) / 128; ++g) {
                    const int b0 = 4 * lane + 128 * g;  // bins b0 .. b0+3 (<= NB - 2); windows cover Lp[b0-4 .. b0+7]
                    const float4 va = *reinterpret_cast<const float4*>(Lp + b0 - 4);
                    const float4 vb = *reinterpret_cast<const float4*>(Lp + b0);
                    const float4 vc = *reinterpret_cast<const float4*>(Lp + b0 + 4);
                    const float4 lc4 = *reinterpret_cast<const float4*>(Lc + b0);
                    // v[0..11] = va.xyzw vb.xyzw vc.xyzw; window of bin b0+j = v[j .. j+8]; common core v[3..8]
                    const float core = fmaxf(fmaxf(fmaxf(va.w, vb.x), fmaxf(vb.y, vb.z)), fmaxf(vb.w, vc.x));
                    const float m0 = fmaxf(fmaxf(core, va.x), fmaxf(va.y, va.z));
                    const float m1 = fmaxf(fmaxf(core, va.y), fmaxf(va.z, vc.y));
                    const float m2 = fmaxf(fmaxf(core, va.z), fmaxf(vc.y, vc.z));
                    const float m3 = fmaxf(fmaxf(core, vc.y), fmaxf(vc.z, vc.w));
                    pair_bin(b0, fmaxf(m0, 0.0f), lc4.x);
                    pair_bin(b0 + 1, fmaxf(m1, 0.0f), lc4.y);
                    pair_bin(b0 + 2, fmaxf(m2, 0.0f), lc4.z);
                    pair_bin(b0 + 3, fmaxf(m3, 0.0f), lc4.w);
                }
                if (lane == 0) {  // the last bin, NB - 1
                    float pm = 0.0f;
                    for (int j = -4; j <= 4; ++j) pm = fmaxf(pm, Lp[NB - 1 + j]);
                    pair_bin(NB - 1, pm, Lc[NB - 1]);
                }
            } else {
                for (int b = lane; b < NB; b += 32) {
                    float pm = 0.0f;
                    for (int j = -K; j <= K; ++j) pm = fmaxf(pm, Lp[b + j]);
                    pair_bin(b, pm, Lc[b]);
                }
            }
        }
        // mel bands (novelty.rs:172-189): the bands' entry lists are cut into 64 chunks of near-equal length (engine.cu), every lane folds two
        // of them in ascending-bin order, then lane m adds the partial sums of band m in order.  One lane per band walked the widest triangle
        // of each round of 32 bands with the other lanes idle (17 % of the kernel's stall samples, ncu r02q; the chunked fold measured 3 % off the
        // kernel); the mel curve only reaches the BPM through tolerance-level novelty values, so the association of the sum is free.
        float* Mc = S.mel[cur];
        const float* Mp = S.mel[cur ^ 1];
        if (nm > 0) {
            const int32_t* ck = st.mel_chunks;
            const int32_t* mbin = st.mel_bin;
            const float* mw = st.mel_w;
#pragma unroll
            for (int r = 0; r < 2; ++r) {
                const int slot = 32 * r + lane;
                const int a = __ldg(ck + slot), e = __ldg(ck + 64 + slot);
                float acc = 0.0f;
                for (int q = a; q < e; ++q) acc = __fadd_rn(acc, __fmul_rn(Lc[__ldg(mbin + q)], __ldg(mw + q)));
                S.part[__ldg(ck + 128 + slot)] = acc;
            }
            __syncwarp();
            for (int m = lane; m < nm; m += 32) {
                float acc = 0.0f;
                for (int j = __ldg(ck + 192 + m); j < __ldg(ck + 193 + m); ++j) acc = __fadd_rn(acc, S.part[j]);
                Mc[m] = acc;
            }
        }
        __syncwarp();
        float ms = 0.0f;
        if (pair) {
            for (int m = lane; m < nm; m += 32) {
                float pmx = 0.0f;
                for (int j = max(m - MK, 0); j < min(m + MK + 1, nm); ++j) pmx = fmaxf(pmx, Mp[j]);
                const float d = fmaxf(Mc[m] - pmx, 0.0f);
                ms += d * d;
            }
        }
        if (emit) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                sf += __shfl_xor_sync(0xffffffffu, sf, o);
                ms += __shfl_xor_sync(0xffffffffu, ms, o);
#pragma unroll
                for (int q = 0; q < 3; ++q) {
                    sfb[q] += __shfl_xor_sync(0xffffffffu, sfb[q], o);
                    Eb[q] += __shfl_xor_sync(0xffffffffu, Eb[q], o);
                    Hb[q] += __shfl_xor_sync(0xffffffffu, Hb[q], o);
                }
            }
            if (lane == 0) {
                for (int q = 0; q < 3; ++q) {
                    fr[(FQ_EB + q) * fm + f] = Eb[q];
                    fr[(FQ_HB + q) * fm + f] = Hb[q];
                }
                if (pair) {
                    pr[PQ_SF * fm + f - 1] = sqrtf(sf);
                    for (int q = 0; q < 3; ++q) pr[(PQ_SFB + q) * fm + f - 1] = sqrtf(sfb[q]);
                    pr[PQ_MEL * fm + f - 1] = sqrtf(ms);
                }
            }
        }
        __syncwarp();
    }
}

// ---- spectral-flux / HFC onsets: exact percentile threshold + peaks -----------------------------
__global__ void __launch_bounds__(256) spectral_onset_kernel(TrackDev* tr, float* fa, int32_t* ia, DevCfg cfg, int which0) {
    __shared__ uint32_t hist[256];
    __shared__ uint32_t bc[2];
    __shared__ uint32_t sc[34];
    TrackDev& T = tr[blockIdx.x];
    const int which = blockIdx.y + which0;  // 0 spectral flux, 1 HFC, 2 HPSS (energy flux of the percussive component, hpss.rs:300-317)
    if (T.status != 0) return;
    if (threadIdx.x == 0) {
        if (which == 0) T.n_on_spectral = 0; else if (which == 1) T.n_on_hfc = 0; else T.n_on_hpss = 0;
    }
    const uint32_t F = T.F[cfg.bs];
    if (F < 2) return;
    const uint32_t L = F - 1;
    const HopLayout& HL = T.hop[cfg.bs];
    const uint64_t fm = HL.fmax;
    const float* flux;
    if (which == 0) {
        flux = fa + HL.pair + PQ_SFLUX * fm;
    } else {
        float* hf = fa + T.scratch + (which == 1 ? fm : 2 * fm);  // HFC flux (hfc.rs:151-154) / percussive energy flux
        const float* H = which == 1 ? fa + HL.frame + FQ_H * fm : fa + T.hop[SLOT_PERC].frame + FQ_E * T.hop[SLOT_PERC].fmax;
        for (uint32_t i = threadIdx.x; i < L; i += blockDim.x) hf[i] = __fadd_rn(fmaxf(__fsub_rn(H[i + 1], H[i]), 0.0f), 0.0f);
        __syncthreads();
        flux = hf;
    }
    uint32_t idx = as_u32(__fmul_rn((float)L, cfg.onset_pct));  // spectral_flux.rs:168
    idx = min(idx, L - 1);
    const float thr = block_select_kth(flux, L, idx, hist, bc);
    int32_t* out = ia + (which == 0 ? T.on_spectral : (which == 1 ? T.on_hfc : T.on_hpss));
    uint32_t total = compact_peaks(flux, L, thr, cfg.hop, T.m, out, sc);  // frame i+1 -> sample (i+1)*hop, kept if < m (lib.rs:181-190)
    if (threadIdx.x == 0) {
        if (which == 0) T.n_on_spectral = total; else if (which == 1) T.n_on_hfc = total; else T.n_on_hpss = total;
    }
}

// ---- consensus vote + caller policy ------------------------------------------------------------
// One CTA per track.  Fast path (lists fit in shared memory): parallel 3-way merge by rank (binary searches,
// method order 0,1,2 on equal samples like the reference's stable sort), gap flags, block scan -> cluster ids,
// one thread per cluster for the integer mean / vote mask, block scan -> compaction (work arrays in global memory beyond CONS_MAX onsets).  Clusters are separated by
// more than `tol` samples, so their centres are strictly increasing and the reference's sort + dedup
// (lib.rs:266-271) is the identity.  Slow path (very long tracks): the same logic run serially by thread 0.
constexpr uint32_t CONS_MAX = 12288;  // onsets (all three lists) handled by the fast path (a 3-minute track has ~5 000)
constexpr uint32_t CONS_SMEM = (CONS_MAX + 2) * 4 + CONS_MAX * (4 + 4) + CONS_MAX + 64;  // in/starts, merged, centres, methods

__device__ __forceinline__ uint32_t count_less(const int32_t* a, uint32_t n, int32_t s, bool or_equal) {
    uint32_t lo = 0, hi = n;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        const bool before = or_equal ? a[mid] <= s : a[mid] < s;
        if (before) lo = mid + 1; else hi = mid;
    }
    return lo;
}

__global__ void __launch_bounds__(256) consensus_kernel(TrackDev* tr, int32_t* ia, float* fa, int n_tracks, DevCfg cfg) {
    extern __shared__ int32_t cs[];
    __shared__ uint32_t sc[34];
    __shared__ uint32_t s_strong;
    const int t = blockIdx.x;
    if (t >= n_tracks) return;
    TrackDev& T = tr[t];
    if (T.status != 0) return;
    const int32_t* G0 = ia + T.on_energy;
    int32_t* gfin = ia + T.on_final;
    const uint32_t n0 = T.n_on_energy;
    if (!cfg.enable_consensus || T.F[cfg.bs] == 0) {
        for (uint32_t i = threadIdx.x; i < n0; i += blockDim.x) gfin[i] = G0[i];
        if (threadIdx.x == 0) T.n_on_final = n0;
        return;
    }
    const int32_t* G1 = ia + T.on_spectral;
    const int32_t* G2 = ia + T.on_hfc;
    const int32_t* G3 = ia + T.on_hpss;
    const uint32_t n1 = T.n_on_spectral, n2 = T.n_on_hfc, n3 = cfg.hpss_onsets ? T.n_on_hpss : 0;
    const uint32_t total = n0 + n1 + n2 + n3;
    if (total == 0) {
        if (threadIdx.x == 0) T.n_on_final = 0;
        return;
    }
    const uint32_t tol = as_u32(__fmul_rn(__fdiv_rn((float)cfg.consensus_tol_ms, 1000.0f), (float)T.sr));  // consensus.rs:149
    // Work arrays: shared memory up to CONS_MAX onsets, else the track's float scratch area in global memory (12 x the largest frame count
    // words; the flux curves it held are dead once the detectors' onset lists exist, and the novelty kernels rewrite it later) — a
    // 60-minute mix has ~32 000 onsets, and the serial fallback below took 41 ms of its 140 ms on one thread (profiles/r02d_bench_c4).
    const bool in_smem = total <= CONS_MAX;
    const uint64_t cap = in_smem ? CONS_MAX : total;
    if (in_smem || (13 * cap) / 4 + 8 <= (uint64_t)12 * T.fall) {
        int32_t* base = in_smem ? cs : reinterpret_cast<int32_t*>(fa + T.scratch);
        int32_t* in = base;                          // [total] the three lists back to back; dead after the merge ...
        int32_t* starts = base;                      // ... and reused as [clusters + 1] first merged index of each cluster
        int32_t* merged = base + cap + 2;            // [total]
        int32_t* centre = base + 2 * cap + 2;        // [clusters] centre; bit 31 marks "voted by >= 2 methods"
        uint8_t* meth = reinterpret_cast<uint8_t*>(base + 3 * cap + 2);  // [total]
        for (uint32_t i = threadIdx.x; i < n0; i += blockDim.x) in[i] = G0[i];
        for (uint32_t i = threadIdx.x; i < n1; i += blockDim.x) in[n0 + i] = G1[i];
        for (uint32_t i = threadIdx.x; i < n2; i += blockDim.x) in[n0 + n1 + i] = G2[i];
        for (uint32_t i = threadIdx.x; i < n3; i += blockDim.x) in[n0 + n1 + n2 + i] = G3[i];
        if (threadIdx.x == 0) s_strong = 0;
        __syncthreads();
        const int32_t* L[4] = {in, in + n0, in + n0 + n1, in + n0 + n1 + n2};
        const uint32_t nl[4] = {n0, n1, n2, n3};
        for (uint32_t e = threadIdx.x; e < total; e += blockDim.x) {
            uint32_t m = 0, i = e;
            while (i >= nl[m]) {
                i -= nl[m];
                ++m;
            }
            const int32_t s = in[e];
            uint32_t r = i;
            for (uint32_t q = 0; q < 4; ++q)
                if (q != m) r += count_less(L[q], nl[q], s, q < m);  // lower method ids come first on ties
            merged[r] = s;
            meth[r] = (uint8_t)m;
        }
        __syncthreads();
        // cluster starts: gap to the previous onset > tol (equivalent to the reference's greedy clustering on a sorted list)
        const uint32_t per = (total + blockDim.x - 1) / blockDim.x;
        const uint32_t a = min(threadIdx.x * per, total), b = min(a + per, total);
        uint32_t cnt = 0;
        for (uint32_t r = a; r < b; ++r) cnt += (r == 0) || ((int64_t)merged[r] - (int64_t)merged[r - 1] > (int64_t)tol);
        uint32_t n_clusters;
        uint32_t pos = block_exclusive_scan(cnt, &n_clusters, sc);
        for (uint32_t r = a; r < b; ++r)
            if ((r == 0) || ((int64_t)merged[r] - (int64_t)merged[r - 1] > (int64_t)tol)) starts[pos++] = (int32_t)r;
        if (threadIdx.x == 0) starts[n_clusters] = (int32_t)total;
        __syncthreads();
        // integer mean + distinct-method count per cluster (consensus.rs:236-262)
        bool any_strong = false;
        for (uint32_t c = threadIdx.x; c < n_clusters; c += blockDim.x) {
            uint64_t sum = 0;
            uint32_t voted = 0;
            const int32_t s0 = starts[c], s1 = starts[c + 1];
            for (int32_t r = s0; r < s1; ++r) {
                sum += (uint64_t)merged[r];
                voted |= 1u << meth[r];
            }
            const bool strong = __popc(voted) >= 2;
            any_strong |= strong;
            centre[c] = (int32_t)(sum / (uint64_t)(s1 - s0)) | (strong ? (int32_t)0x80000000 : 0);  // samples < 2^31: bit 31 is free
        }
        if (any_strong) s_strong = 1;  // benign race: every writer stores 1
        __syncthreads();
        const bool want_strong = s_strong != 0;  // lib.rs:258-271: clusters voted by >= 2 methods, else all of them
        const uint32_t perc = (n_clusters + blockDim.x - 1) / blockDim.x;
        const uint32_t ca = min(threadIdx.x * perc, n_clusters), cb = min(ca + perc, n_clusters);
        uint32_t keep = 0;
        for (uint32_t c = ca; c < cb; ++c) keep += !want_strong || (centre[c] < 0);
        uint32_t nfinal;
        uint32_t w = block_exclusive_scan(keep, &nfinal, sc);
        for (uint32_t c = ca; c < cb; ++c)
            if (!want_strong || (centre[c] < 0)) gfin[w++] = centre[c] & 0x7fffffff;
        if (threadIdx.x == 0) T.n_on_final = nfinal;
        return;
    }
    // ---- slow path ----
    if (threadIdx.x == 0) {
        const int32_t *L0 = G0, *L1 = G1, *L2 = G2, *L3 = G3;
        int32_t* fin = gfin;
        uint32_t strong = 0, nfinal = 0;
        for (int pass = 0; pass < 2; ++pass) {
            const bool want_strong = strong > 0;
            uint32_t i0 = 0, i1 = 0, i2 = 0, i3 = 0, w = 0;
            bool open = false;
            int64_t last = 0;
            uint64_t sum = 0;
            uint32_t cnt = 0, voted = 0;
            auto close = [&]() {
                const int32_t c = (int32_t)(sum / cnt);
                const uint32_t vb = __popc(voted);
                if (pass == 0) {
                    if (vb >= 2) ++strong;
                } else if (!want_strong || vb >= 2) {
                    if (w == 0 || fin[w - 1] != c) fin[w++] = c;
                }
            };
            while (i0 < n0 || i1 < n1 || i2 < n2 || i3 < n3) {
                int method = -1;
                int32_t s = 0x7fffffff;
                if (i0 < n0 && L0[i0] < s) { s = L0[i0]; method = 0; }
                if (i1 < n1 && L1[i1] < s) { s = L1[i1]; method = 1; }
                if (i2 < n2 && L2[i2] < s) { s = L2[i2]; method = 2; }
                if (i3 < n3 && L3[i3] < s) { s = L3[i3]; method = 3; }
                if (method == 0) ++i0; else if (method == 1) ++i1; else if (method == 2) ++i2; else ++i3;
                if (open && (int64_t)s - last > (int64_t)tol) { close(); open = false; }
                if (!open) { open = true; sum = 0; cnt = 0; voted = 0; }
                sum += (uint64_t)s;
                ++cnt;
                voted |= 1u << method;
                last = s;
            }
            if (open) close();
            if (pass == 1) nfinal = w;
        }
        T.n_on_final = nfinal;
    }
}

void launch_energy_onsets(const WaveCtx& c) {
    if (c.max_F[c.cfg.bs] > 0) {
        with_frame(c.cfg.frame, [&](auto fc) {
            constexpr int FR = decltype(fc)::F, PER_CTA = ERMS_SEG * 4 * ERMS_GPW<FR>;  // frames per CTA of the streamed form
            if (c.cfg.bs == 0) energy_rms_kernel<FR><<<dim3((c.max_F[0] + PER_CTA - 1) / PER_CTA, c.n_tracks), 128, 0, c.stream>>>(c.samples, c.tracks, c.fa);
            else energy_rms_any_kernel<FR><<<dim3((c.max_F[c.cfg.bs] + 127) / 128, c.n_tracks), 128, 0, c.stream>>>(c.samples, c.tracks, c.fa, c.cfg.hop, c.cfg.bs);
        });
        count_launch("onsets");
    }
    energy_onset_kernel<<<c.n_tracks, 256, 0, c.stream>>>(c.tracks, c.fa, c.ia, c.cfg);
    count_launch("onsets");
}

// Percussive-component onsets (lib.rs:222-235): frame energies come from seq_feat_kernel on the percussive slot.
void launch_hpss_onsets(const WaveCtx& c) {
    if (c.max_F[c.cfg.bs] == 0) return;
    spectral_onset_kernel<<<dim3(c.n_tracks, 1), 256, 0, c.stream>>>(c.tracks, c.fa, c.ia, c.cfg, 2);
    count_launch("hpss");
}

static void launch_seq(const WaveCtx& c, int h, const int32_t* d_list, int n_list) {
    const dim3 grid((c.max_F[h] + 123) / 124, n_list);  // 4 warps x 31 new frames
    with_frame(c.cfg.frame, [&](auto fc) {
        constexpr int NB = decltype(fc)::B;
        if (h == 1) seq_feat_kernel<1, NB><<<grid, 128, 0, c.stream>>>(c.tracks, d_list, h, c.fa);
        else if (h == 2) seq_feat_kernel<2, NB><<<grid, 128, 0, c.stream>>>(c.tracks, d_list, h, c.fa);
        else seq_feat_kernel<0, NB><<<grid, 128, 0, c.stream>>>(c.tracks, d_list, h, c.fa);
    });
    count_launch("spec_features");
}

void launch_seq_features(const WaveCtx& c, int h, const int32_t* d_list, int n_list) {
    if (c.max_F[h] == 0 || n_list == 0) return;
    launch_seq(c, h, d_list, n_list);
}

template <bool K4, int MODE, int NB>
static void launch_par_mode(const WaveCtx& c, int h, const int32_t* d_list, int n_list) {
    constexpr int W = PAR_WARPS<NB>;
    constexpr size_t smem = NB == 1025 ? 0 : W * sizeof(ParSmem<NB>);
    if (smem > 0) {
        static bool attr_dev[64] = {};  // function attributes are per device
        int dev = 0;
        cudaGetDevice(&dev);
        if (!attr_dev[dev & 63]) {
            cudaFuncSetAttribute(par_feat_kernel<K4, MODE, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            attr_dev[dev & 63] = true;
        }
    }
    const dim3 grid((c.max_F[h] + W * FEAT_RUN - 1) / (W * FEAT_RUN), n_list);
    par_feat_kernel<K4, MODE, NB><<<grid, 32 * W, smem, c.stream>>>(c.tracks, d_list, c.srtab, c.sr_index, h, c.fa, c.cfg);
}

template <bool K4>
static void launch_par(const WaveCtx& c, int h, const int32_t* d_list, int n_list) {
    with_frame(c.cfg.frame, [&](auto fc) {
        constexpr int NB = decltype(fc)::B;
        if (h == 1) launch_par_mode<K4, 1, NB>(c, h, d_list, n_list);
        else if (h == 2) launch_par_mode<K4, 2, NB>(c, h, d_list, n_list);
        else launch_par_mode<K4, 0, NB>(c, h, d_list, n_list);
    });
    count_launch("spec_features");
}

void launch_spec_features(const WaveCtx& c, int h, const int32_t* d_list, int n_list) {
    if (c.max_F[h] == 0 || n_list == 0) return;
    launch_seq(c, h, d_list, n_list);
    if (std::min(std::max(c.cfg.sf_k, 1u), (uint32_t)HALO) == 4u) launch_par<true>(c, h, d_list, n_list);
    else launch_par<false>(c, h, d_list, n_list);
}

void launch_spectral_onsets_consensus(const WaveCtx& c) {
    if (c.cfg.enable_consensus && c.max_F[c.cfg.bs] > 0) {
        spectral_onset_kernel<<<dim3(c.n_tracks, 2), 256, 0, c.stream>>>(c.tracks, c.fa, c.ia, c.cfg, 0);
        count_launch("onsets");
    }
    {
        static bool attr_dev[64] = {};  // function attributes are per device
        int dev = 0;
        cudaGetDevice(&dev);
        if (!attr_dev[dev & 63]) {
            cudaFuncSetAttribute(consensus_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, CONS_SMEM);
            attr_dev[dev & 63] = true;
        }
    }
    consensus_kernel<<<c.n_tracks, 256, CONS_SMEM, c.stream>>>(c.tracks, c.ia, c.fa, c.n_tracks, c.cfg);
    count_launch("onsets");
}

}  // namespace sb
