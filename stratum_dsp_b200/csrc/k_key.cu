// Key detection kernels — the default key path of analyze_audio (reference lib.rs:961-1559):
//   soft harmonic time mask            chroma/extractor.rs:1246-1349   (mask_kernel, in place)
//   HPCP per frame + frame energy      chroma/extractor.rs:529-680, 1097-1150 (hpcp_kernel)
//   5-tap median smoothing             chroma/smoothing.rs:37-94       (chroma_smooth_kernel)
//   tonalness / energy frame weights   lib.rs:1236-1287                (key_weights_kernel)
//   segment template scores            key/detector.rs:118-133, 984-1001 (segment_score_kernel)
//   normalise, circle-of-fifths bonus, ranking, clarity, clarity-weighted vote
//                                      key/detector.rs:135-313, key_clarity.rs:51-93, lib.rs:1332-1436 (key_vote_kernel)
//
// HBM traffic per key frame: the 4097-bin magnitude row is written once by the STFT, read + rewritten
// in place by the mask and read once by the HPCP kernel (4 x 16 KB); everything after that is 12 floats
// per frame.
#include <type_traits>

#include "framed.cuh"
#include "key_rows.cuh"

namespace sb {

constexpr int RING = 32;           // mask ring: supports margin <= 15
constexpr int HPCP_PEAKS_44K = 512;   // local maxima in the 100..5000 Hz band: <= (hi-lo+2)/2 = 456 at 44.1 kHz, 420 at 48 kHz
constexpr int HPCP_PEAKS_ANY = 2048;  // any sample rate: a row of the 8192-point key STFT has at most 4097 / 2 local maxima
constexpr int HPCP_MAX_SEL = 32;     // key_hpcp_peaks_per_frame upper bound accepted by the ABI
constexpr int HPCP_MAX_HARM = 8;     // key_hpcp_num_harmonics upper bound accepted by the ABI

// ---- soft harmonic mask: one thread per (track, bin), strictly sequential f32 prefix over time ----
// The reference builds `prefix[t+1] = prefix[t] + x[t]` per bin and takes window sums as prefix
// differences (extractor.rs:1274-1287); the cancellation noise of that formulation is part of its
// output, so the scan is reproduced term by term.  Adjacent threads own adjacent bins, so every
// load and store of a frame row is coalesced.  Frames are consumed in half-steps of 8 whose loads are
// issued one half-step ahead (see the frame loop); stores only touch rows already consumed, so the
// non-compact variant writes the mask in place.  MG > 0: margin known at compile time, the delayed sample
// x[t - MG] is then a register; MG = 0: run-time margin with a shared-memory ring for the samples.
constexpr int MASK_G = 16;

// FAST: the default exponent 2 with the mask on — `h*h`, `r*r` and no per-element mode tests.
// KB: bins per key-spectrogram row when known at compile time (4097 for the default 8192-point key STFT: row offsets become
// immediates), 0 = cfg.key_bins.
// COMPACT: the masked rows are read again only by the HPCP peak search (bins [kband_lo, kband_lo + kband_stride)) and through the
// frame energy sum(y^2) over all bins, so instead of rewriting the 16 KB row in place the kernel writes the band columns into the
// compact buffer T.kband [Fk x kband_stride] and each WARP's 32-bin share of every frame's energy into T.kepart[warp][t]
// (hpcp_kernel adds the shares in warp order).  The spectrogram is then read exactly once and 78 % of the mask's stores and of the
// HPCP kernel's loads disappear.  The shares go through a per-warp shared tile [16 frames x 32 bins (+1 pad)] folded after each
// 16-frame group: lane l sums 16 bins of frame l mod 16, one shuffle joins the two halves — about 35 instructions per thread and
// group, off the per-element chain, and no CTA barrier (a first version with a CTA-wide tile and one barrier per group ran 38 %
// slower than the in-place kernel: the barrier serialises the four warps' load latencies).
// BS: floats per row of the compact band when known at compile time (960 covers the 100..5000 Hz band of the 8192-point key STFT at every
// sample rate >= 39.2 kHz: the band stores become base + immediate instead of a 64-bit multiply-add per element), 0 = T.kband_stride.
// Two 16-frame groups per loop trip: the prefix ring has 32 slots, so with the trip starting at a multiple of 32 every ring index of the
// steady state is a compile-time constant (ncu/SASS of the one-group loop: five uniform-datapath instructions per element rebuilding
// (ii & 31) * 512 offsets, six for the band store's address — 37 instructions per element, 24 of them arithmetic).
// seg_len > 0 (COMPACT only, a multiple of 32): the track is cut into floor(Fk / seg_len) time segments, one per blockIdx.z, for waves with
// too few tracks to fill the device (a single 60-minute mix is 33 CTAs walking 310 000 frames each: 36 ms on 3 % of the warps).  Segment z
// starts from the exact prefix of the frames before z * seg_len (mask_prefix_kernel: the same serial additions, nothing else), consumes
// frames [z * seg_len, (z + 1) * seg_len + 32) and emits every frame whose window it has seen in full — the 20 frames two neighbouring
// segments both emit get bit-identical values.  Only the last segment runs the tail and the flush.
// Seven CTAs per SM (72 registers): under the nine-CTA cap of 56 registers the compiler could not overlap the dependent chains of
// neighbouring frames; per 512 tracks (r02D-r02G) 9 CTAs 53.5 ms, 8 CTAs 51.9, 7 CTAs 41.1, 6 CTAs 43.5, 5 CTAs 48.2.
template <int MG, bool FAST, int KB, bool COMPACT, int BS = 0>
__global__ void __launch_bounds__(128, 7) mask_kernel(const TrackDev* __restrict__ tr, float* fa, DevCfg cfg, uint32_t seg_len) {
    const uint32_t KBINS = KB ? (uint32_t)KB : cfg.key_bins;
    // floats per spectrogram row: the compact variant's input rows are padded to a 32-byte sector by the STFT (DevCfg::key_stride), so a
    // warp's 128-byte load is four aligned sectors instead of five (ncu: 309 MB read per track for 254 MB of rows before the padding)
    const uint32_t KSTRIDE = COMPACT ? (KB ? (uint32_t)((KB + 7) / 8 * 8) : cfg.key_stride) : KBINS;
    __shared__ float ringP[RING][128];
    __shared__ float ringX[MG > 0 ? 1 : RING][128];
    __shared__ float et[COMPACT ? 4 : 1][COMPACT ? MASK_G : 1][COMPACT ? 33 : 1];
    const TrackDev& T = tr[blockIdx.y];
    const uint32_t nf = T.Fk;
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = b < KBINS;
    if (T.status != 0 || nf == 0) return;
    const int tx = threadIdx.x;
    const int wid = tx >> 5, lane = tx & 31;
    if (blockIdx.x * blockDim.x + (uint32_t)wid * 32u >= KBINS) return;  // whole warp past the row
    if (!COMPACT && !valid) return;  // the compact variant has warp collectives in the frame loop: idle lanes run it on zeros
    const uint32_t mg = MG > 0 ? (uint32_t)MG : cfg.key_margin;
    float* K = fa + T.keyspec + (valid ? b : 0u);
    const bool inband = COMPACT && valid && b >= T.kband_lo && b < T.kband_lo + T.kband_stride;
    float* B = fa + T.kband + (inband ? b - T.kband_lo : 0u);
    const uint32_t bstride = BS ? (uint32_t)BS : T.kband_stride;
    float* EP = fa + T.kepart + (uint64_t)(blockIdx.x * 4 + wid) * T.kepart_stride;  // this warp's share row
    const float p = FAST ? 2.0f : fmaxf(cfg.key_mask_power, 1.0f);
    const bool square = FAST || (p == 2.0f);
    const uint32_t z = COMPACT ? blockIdx.z : 0u;
    const uint32_t nz = (COMPACT && seg_len) ? max(1u, nf / seg_len) : 1u;
    if (z >= nz) return;
    const uint32_t c0 = z * seg_len;                                    // first frame consumed (a multiple of the ring length)
    const bool last = z + 1 == nz;
    const uint32_t c1 = last ? nf : c0 + seg_len + RING;                // one past the last frame consumed
    const uint32_t emit_from = z ? c0 + 2 * mg : mg;                    // frame t = ii - mg is emitted for consumed frames ii >= emit_from
    float P = (z && valid) ? fa[T.kprefix + (uint64_t)(z - 1) * KSTRIDE + b] : 0.0f;  // prefix[c0]
    ringP[0][tx] = P;
    auto ld = [&](uint32_t t) { return (!COMPACT || valid) ? K[(uint64_t)t * KSTRIDE] : 0.0f; };
    // where frame t's masked value goes: its column of the compact band, or the spectrogram row itself (in place)
    const uint32_t dstride = COMPACT ? bstride : KSTRIDE;
    float* const D = COMPACT ? B : K;
    auto dst_of = [&](uint32_t t) { return D + (uint64_t)t * dstride; };
    // row >= 0: slot of the warp's energy tile this frame's share goes to (16-frame groups); row < 0: the tail, folded per frame
    auto put = [&](uint32_t t, float* dst, float y, int row) {
        if (!COMPACT) {
            *dst = y;
            return;
        }
        if (inband) *dst = y;
        const float e = y * y;
        if (row >= 0) {
            et[wid][row][lane] = e;
        } else {  // warp-wide fold of one frame (uniform control flow: every lane emits the same frames)
            float v = e;
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == 0) EP[t] = v;
        }
    };
    // steady = the window [t - mg, t + mg] lies inside the track: the divisor is the compile-time constant 2*MG + 1 (an IEEE
    // division by a constant needs no reciprocal approximation or range check), no clamping of the window edges
    auto emit_h = [&](uint32_t t, float* dst, float h_est, float xt, int row) {
        if (!FAST && cfg.key_smooth_only) {  // smooth_spectrogram_time alone (extractor.rs:1246-1290, lib.rs:1043-1060)
            put(t, dst, h_est, row);
            return;
        }
        const float x = fmaxf(xt, 0.0f);
        const float h = fmaxf(h_est, 0.0f);
        const float r = fmaxf(x - h, 0.0f);
        const float hp = square ? h * h : powf(h, p);
        const float rp = square ? r * r : powf(r, p);
        // FAST: hp, rp are squares of magnitudes (<= 2^40) and the divisor is >= 1e-12, so the quotient is correctly rounded
        // without the generic division's range check (common.cuh); hp below 2^-100 only occurs below -600 dBFS
        const float m = FAST ? div_rn_inrange(hp, hp + rp + 1e-12f) : hp / (hp + rp + 1e-12f);
        put(t, dst, x * m, row);
    };
    auto emit = [&](uint32_t t, float* dst, uint32_t en, float Pen, float xt, int row) {
        float h_est;
        if (mg == 0) {
            h_est = xt;
        } else {
            const uint32_t st = t >= mg ? t - mg : 0;
            const float sum = Pen - ringP[st & (RING - 1)][tx];
            const float denom = (float)max(en - st, 1u);
            h_est = sum / denom;
        }
        emit_h(t, dst, h_est, xt, row);
    };
    // The main part of the track (whole 16-frame groups) runs as half-steps of 8 frames over four register arrays in rotating roles:
    // step k consumes h[k & 3] (frames 8k .. 8k+7), takes its delayed samples x[t - MG] from the two arrays before it, and starts the
    // loads of step k + 1 into the fourth BEFORE it computes — so every load has a whole half-step of arithmetic (~240 instructions per
    // warp, times the other resident warps) to land, with the same 32 sample registers the one-group form used for "this group" and
    // "previous group".  (r02q/r02r: with the loads issued at the top of the group that consumes them the kernel sat on the long
    // scoreboard for 22 % of its samples, and 19 % fewer instructions did not move its run time.)  R = k & 3 and STEADY are types:
    // four steps per loop trip make every prefix-ring slot a compile-time constant, and the clipped-window code of the first ring
    // revolution stays out of the steady loop.
    constexpr int H = 8;
    static_assert(RING == 4 * H && MASK_G == 2 * H, "four half-steps per ring revolution, two per energy tile");
    static_assert(MG == 0 || (MG > H && MG <= 2 * H), "delayed samples come from the two previous half-steps");
    float h[4][H];
#pragma unroll
    for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int q = 0; q < H; ++q) h[r][q] = 0.0f;
    const uint32_t k0 = c0 / H, k_end = k0 + 2 * ((c1 - c0) / MASK_G);
    const float* kp = K + (uint64_t)c0 * KSTRIDE;                              // row 8k of this thread's column
    float* dp = D + ((int64_t)c0 - (int64_t)mg) * (int64_t)dstride;            // destination of frame 8k - mg; only dereferenced for emitted frames
    auto fetch = [&](float (&dst)[H], const float* from) {
#pragma unroll
        for (int q = 0; q < H; ++q) dst[q] = (!COMPACT || valid) ? from[(uint32_t)q * KSTRIDE] : 0.0f;
    };
    auto step = [&](uint32_t k, auto r_t, auto st) {
        constexpr int R = decltype(r_t)::value;
        constexpr bool steady = MG > 0 && decltype(st)::value;
        const uint32_t i = k * H;
        if (k + 1 < k_end) fetch(h[(R + 1) & 3], kp + (uint64_t)H * KSTRIDE);
        const float(&cur)[H] = h[R];
        const float(&p1)[H] = h[(R + 3) & 3];
        const float(&p2)[H] = h[(R + 2) & 3];
#pragma unroll
        for (int q = 0; q < H; ++q) {
            const uint32_t ii = i + q;
            constexpr int PH = R * H;
            const int row = (R & 1) * H + q;  // slot of the warp's 16-frame energy tile
            if (MG == 0) ringX[(PH + q) & (RING - 1)][tx] = cur[q];
            P = P + cur[q];
            if (steady || ii >= emit_from) {  // prefix[t - mg] was written 2*mg+1 steps ago: still in the ring
                float xt;
                if (MG > 0) xt = (q + 2 * H - MG < H) ? p2[(q + 2 * H - MG) & (H - 1)] : p1[(q + H - MG) & (H - 1)];  // x[8k + q - MG]
                else xt = ringX[(ii - mg) & (RING - 1)][tx];
                if (steady) {
                    const float wsum = P - ringP[(PH + q + 2 * RING - 2 * MG) & (RING - 1)][tx];
                    // FAST (mask on, margin 12): RN(wsum / 25) in three instructions; exact for |wsum| >= 1e-30, and a smaller window sum
                    // gives h < 1e-31, whose square is zero whichever way the quotient rounds
                    emit_h(ii - MG, dp + (uint32_t)q * dstride, (FAST && MG == 12) ? div_by_25_rn(wsum) : wsum / (float)(2 * MG + 1), xt, row);
                }
                else emit(ii - mg, dp + (uint32_t)q * dstride, ii + 1, P, xt, row);
            }
            ringP[(PH + q + 1) & (RING - 1)][tx] = P;
        }
        kp += (uint64_t)H * KSTRIDE;
        dp += (uint64_t)H * dstride;
        if (COMPACT && (R & 1)) {  // fold the warp's tile: lane l adds bins 16*(l/16) .. +15 of row l % 16 (frame i16 + row - mg), halves joined by one shuffle
            const uint32_t i16 = i - H;
            __syncwarp();
            const int row = lane & (MASK_G - 1), c0 = (lane >> 4) * 16;
            float v = 0.0f;
#pragma unroll
            for (int c = 0; c < 16; ++c) v += et[wid][row][c0 + c];
            v += __shfl_xor_sync(0xffffffffu, v, 16);
            if (lane < MASK_G && (steady || i16 + row >= emit_from)) EP[i16 + row - mg] = v;
            __syncwarp();
        }
    };
    using R0 = std::integral_constant<int, 0>;
    using R1 = std::integral_constant<int, 1>;
    using R2 = std::integral_constant<int, 2>;
    using R3 = std::integral_constant<int, 3>;
    uint32_t k = k0;
    if (k_end > k0) fetch(h[0], kp);
    if (k_end - k0 >= 4) {  // first ring revolution: windows clipped at the track start / frames before the segment's first full window
        step(k, R0{}, std::false_type{});
        step(k + 1, R1{}, std::false_type{});
        step(k + 2, R2{}, std::false_type{});
        step(k + 3, R3{}, std::false_type{});
        k += 4;
    }
    for (; k + 4 <= k_end; k += 4) {
        step(k, R0{}, std::true_type{});
        step(k + 1, R1{}, std::true_type{});
        step(k + 2, R2{}, std::true_type{});
        step(k + 3, R3{}, std::true_type{});
    }
    if (k + 2 <= k_end) {  // one more group of 16
        if (k == k0) {
            step(k, R0{}, std::false_type{});
            step(k + 1, R1{}, std::false_type{});
        } else {
            step(k, R0{}, std::true_type{});
            step(k + 1, R1{}, std::true_type{});
        }
        k += 2;
    }
    if (!last) return;
    uint32_t i = k * H;
    // tail (< 16 frames) and flush: the delayed samples are re-read from rows that are still unmasked
    // (row t is only rewritten by emit(t)), which costs at most 16 + margin scalar loads per thread
    for (; i < nf; ++i) {
        const float x = ld(i);
        P = P + x;
        if (i >= emit_from) emit(i - mg, dst_of(i - mg), i + 1, P, ld(i - mg), -1);
        ringP[(i + 1) & (RING - 1)][tx] = P;
    }
    for (uint32_t t = max(nf > mg ? nf - mg : 0u, z ? c0 + mg : 0u); t < nf; ++t) emit(t, dst_of(t), nf, P, ld(t), -1);
}

// Exact prefixes at the segment starts of a time-segmented mask launch: prefix[z - 1][bin] = the serial f32 sum of the bin's magnitudes
// over frames [0, z * seg_len), z = 1 .. nz - 1 — the additions of the mask's own scan and nothing else, so a segment that starts from it
// continues the reference's rounding sequence (extractor.rs:1274-1279).  A pure dependent add chain per thread; the rows are fetched 48
// frames ahead (three register batches of 16 in flight) because with one warp per scheduler nothing else hides the memory latency.
template <int KB>
__global__ void __launch_bounds__(128) mask_prefix_kernel(const TrackDev* __restrict__ tr, float* fa, DevCfg cfg, uint32_t seg_len) {
    const uint32_t KBINS = KB ? (uint32_t)KB : cfg.key_bins;
    const uint32_t KSTRIDE = KB ? (uint32_t)((KB + 7) / 8 * 8) : cfg.key_stride;
    const TrackDev& T = tr[blockIdx.y];
    const uint32_t nf = T.Fk;
    const uint32_t b = blockIdx.x * blockDim.x + threadIdx.x;
    if (T.status != 0 || b >= KBINS || seg_len == 0) return;
    const uint32_t nz = max(1u, nf / seg_len);
    if (nz < 2) return;
    const float* K = fa + T.keyspec + b;
    float* out = fa + T.kprefix + b;
    const uint32_t per_seg = seg_len / 16;          // seg_len is a multiple of 32
    const uint32_t n_batches = (nz - 1) * per_seg;
    float a[4][16];
    auto fetch = [&](float (&dst)[16], uint32_t batch) {
        const float* p = K + (uint64_t)batch * 16 * KSTRIDE;
#pragma unroll
        for (int q = 0; q < 16; ++q) dst[q] = p[(uint32_t)q * KSTRIDE];
    };
    fetch(a[0], 0);
    if (n_batches > 1) fetch(a[1], 1);
    if (n_batches > 2) fetch(a[2], 2);
    float P = 0.0f;
    auto consume = [&](uint32_t j, auto r_t) {
        constexpr int R = decltype(r_t)::value;
        if (j + 3 < n_batches) fetch(a[(R + 3) & 3], j + 3);
#pragma unroll
        for (int q = 0; q < 16; ++q) P = P + a[R][q];
        if ((j + 1) % per_seg == 0) out[(uint64_t)((j + 1) / per_seg - 1) * KSTRIDE] = P;
    };
    uint32_t j = 0;
    for (; j + 4 <= n_batches; j += 4) {
        consume(j, std::integral_constant<int, 0>{});
        consume(j + 1, std::integral_constant<int, 1>{});
        consume(j + 2, std::integral_constant<int, 2>{});
        consume(j + 3, std::integral_constant<int, 3>{});
    }
    if (j < n_batches) consume(j++, std::integral_constant<int, 0>{});
    if (j < n_batches) consume(j++, std::integral_constant<int, 1>{});
    if (j < n_batches) consume(j++, std::integral_constant<int, 2>{});
}

// ---- HPCP: one warp per frame ---------------------------------------------------------------------
// MAXI: (peak, harmonic) items per frame the instantiation has room for (the defaults need 24 x 4 = 96)
template <int MAXP, int MAXI = HPCP_MAX_SEL * HPCP_MAX_HARM>
struct HpcpSmem {
    float mag[MAXP];
    uint16_t bin[MAXP];
    uint16_t sel[HPCP_MAX_SEL];
    // per (peak, harmonic) item: val[4 it + s], s = 1..3 = its contributions to the pitch classes primary - 1, primary, primary + 1
    // (slot 0 = 0.0f), and map[it] = twelve 2-bit slot numbers, class c at bits 2c (0 = no contribution)
    __align__(16) float val[MAXI * 4];
    __align__(16) uint32_t map[MAXI];
};

__device__ __forceinline__ float rem_euclid_f(float a, float b) {
    float r = fmodf(a, b);
    return r < 0.0f ? r + fabsf(b) : r;
}

// One band of frame_to_hpcp_tuned_band (extractor.rs:529-680) for the calling warp.  `sel` = the row peaks are picked and ranked
// on (whitened magnitudes when whitening is on, else the magnitudes), `mag` = the magnitudes that weight the peaks.
// Returns the L2-normalised profile in lanes 0..11.
template <int MAXP, int MAXI>
__device__ __forceinline__ float hpcp_band(const float* __restrict__ sel, const float* __restrict__ mag, uint32_t lo, uint32_t hi, float fmin, float fmax,
                                           uint32_t peaks_per_frame, float tuning, float res, HpcpSmem<MAXP, MAXI>& S, int lane, const DevCfg& cfg) {
    constexpr int HPCP_MAX_PEAKS = MAXP;
    // local maxima in the band, compacted in ascending bin order (extractor.rs:582-606)
    // Eight 32-bin slices at a time: their values are fetched first (eight independent loads in flight instead of three
    // dependent ones per slice), neighbours come from the adjacent lanes / slices by shuffle, then the compare-ballot-compact
    // chain runs on registers.
    uint32_t np = 0;
    if (lo <= hi) {
        for (uint32_t base0 = lo; base0 <= hi; base0 += 256) {
            float mv[8];
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t b = base0 + 32 * k + lane;
                mv[k] = b <= hi + 1 ? sel[b] : 0.0f;  // hi + 1 is a valid bin (the band loop stops two bins short of the row end)
            }
            const float left_edge = sel[base0 - 1];
            const float right_edge = base0 + 256 <= hi + 1 ? sel[base0 + 256] : 0.0f;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const uint32_t b = base0 + 32 * k + lane;
                const float m = mv[k];
                float l = __shfl_up_sync(0xffffffffu, m, 1);
                const float lc = k == 0 ? left_edge : __shfl_sync(0xffffffffu, mv[k > 0 ? k - 1 : 0], 31);
                if (lane == 0) l = lc;
                float r = __shfl_down_sync(0xffffffffu, m, 1);
                const float rc = k == 7 ? right_edge : __shfl_sync(0xffffffffu, mv[k < 7 ? k + 1 : 7], 0);
                if (lane == 31) r = rc;
                const bool pk = b <= hi && !(m <= l || m < r);
                const uint32_t mask = __ballot_sync(0xffffffffu, pk);
                if (pk) {
                    const uint32_t pos = np + __popc(mask & ((1u << lane) - 1u));
                    if (pos < HPCP_MAX_PEAKS) {
                        S.mag[pos] = m;
                        S.bin[pos] = (uint16_t)b;
                    }
                }
                np += __popc(mask);
            }
        }
        np = min(np, (uint32_t)HPCP_MAX_PEAKS);
    }
    __syncwarp();
    float pc = 0.0f;  // lanes 0..11 own one pitch class each
    if (np > 0) {
        // top-K by (value desc, bin asc); the reference's select_nth_unstable_by leaves the K
        // survivors in unspecified order — the documented rule is "accumulate in ascending bin order".
        // The K-th largest value is found by a bitwise search on the (positive) float bit patterns:
        // 31 rounds of "how many peaks are >= candidate", each a register compare + one warp reduction.
        const uint32_t K = min(max(peaks_per_frame, 1u), np);
        uint32_t thr = 0, need = 0;  // keep values > thr, plus the first `need` ties in bin order
        if (np > K) {
            uint32_t e[HPCP_MAX_PEAKS / 32];
#pragma unroll
            for (int q = 0; q < HPCP_MAX_PEAKS / 32; ++q) {
                const uint32_t i = q * 32 + lane;
                e[q] = i < np ? __float_as_uint(S.mag[i]) : 0u;  // peaks are strictly positive, 0 never counts
            }
            // Early exit: as soon as exactly K values are >= cand the survivors are known (everything >= cand) whatever the lower bits of
            // the K-th value are, so the search stops with thr = cand - 1 ("> thr" == ">= cand", and values equal to thr are then
            // offered as ties with need = 0).  The K-th and (K+1)-th largest peaks of a spectrum row rarely share more than the exponent
            // and a few mantissa bits: about a dozen rounds instead of 31, same selection.
            for (int bit = 30; bit >= 0; --bit) {
                const uint32_t cand = thr | (1u << bit);
                uint32_t c = 0;
#pragma unroll
                for (int q = 0; q < HPCP_MAX_PEAKS / 32; ++q) c += e[q] >= cand;
                c = __reduce_add_sync(0xffffffffu, c);
                if (c == K) {
                    thr = cand - 1u;
                    break;
                }
                if (c > K) thr = cand;
            }
            uint32_t gt = 0;
#pragma unroll
            for (int q = 0; q < HPCP_MAX_PEAKS / 32; ++q) gt += e[q] > thr;
            need = K - __reduce_add_sync(0xffffffffu, gt);
        }
        uint32_t nsel = 0, ties_seen = 0;
        for (uint32_t base = 0; base < np; base += 32) {
            const uint32_t i = base + lane;
            bool keep = false, tie = false;
            if (i < np) {
                if (np <= K) {
                    keep = true;
                } else {
                    const uint32_t bits = __float_as_uint(S.mag[i]);
                    keep = bits > thr;
                    tie = bits == thr;
                }
            }
            const uint32_t tmask = __ballot_sync(0xffffffffu, tie);
            if (tie && ties_seen + __popc(tmask & ((1u << lane) - 1u)) < need) keep = true;
            ties_seen += __popc(tmask);
            const uint32_t mask = __ballot_sync(0xffffffffu, keep);
            if (keep) S.sel[nsel + __popc(mask & ((1u << lane) - 1u))] = (uint16_t)i;
            nsel += __popc(mask);
        }
        __syncwarp();
        const float sigma = fmaxf(cfg.hpcp_sigma, 1e-6f);
        const uint32_t hmax = min(max(cfg.hpcp_harm, 1u), (uint32_t)HPCP_MAX_HARM);
        const float decay = clamp_rs(cfg.hpcp_decay, 0.0f, 1.0f);
        const float pw = clamp_rs(cfg.hpcp_pow, 0.05f, 1.0f);
        const uint32_t items = nsel * hmax;
        for (uint32_t it = lane; it < items; it += 32) {
            const uint32_t pi = it / hmax, h = it % hmax + 1;
            const uint32_t idx = S.sel[pi];
            const uint32_t bin = S.bin[idx];
            const float f0 = (float)bin * res;
            const float mg = fmaxf(mag[bin], 0.0f);  // the original magnitude weights the peak even when whitening picked it (:628-637)
            const float w0 = (pw == 0.5f) ? sqrtf(mg) : powf(mg, pw);
            const float fh = f0 * (float)h;
            float* vals = S.val + it * 4;
            vals[0] = 0.0f;
            // `break` at fh > fmax and `continue` at fh < fmin both leave this (peak, h) without a contribution
            if (!(f0 > 0.0f) || !(w0 > 0.0f) || fh > fmax || fh < fmin) {
                S.map[it] = 0u;
                continue;
            }
            const float semitone = 12.0f * log2f(fh / 440.0f) + 57.0f - tuning;
            const float spc = rem_euclid_f(semitone, 12.0f);
            const float ppc = rem_euclid_f(roundf(spc), 12.0f);
            const int primary = as_i32(ppc);
            float dp = 1.0f, da = decay;  // decay.powi(h - 1) as compiler-rt's __powisf2 evaluates it: square-and-multiply
            for (uint32_t e = h - 1;;) {
                if (e & 1u) dp = dp * da;
                e >>= 1;
                if (e == 0) break;
                da = da * da;
            }
            const float hw = dp / (float)h;
            const float contrib = w0 * hw;
            uint32_t map = 0u;
#pragma unroll
            for (int off = -1; off <= 1; ++off) {
                const int tc = ((primary + off) % 12 + 12) % 12;
                float dist = fabsf(spc - (float)tc);
                dist = fminf(dist, 12.0f - dist);
                const float wgt = expf(-dist * dist / (2.0f * sigma * sigma));
                map |= (uint32_t)(off + 2) << (2 * tc);  // the three classes are distinct
                vals[off + 2] = contrib * wgt;
            }
            S.map[it] = map;
        }
        const uint32_t items4 = (items + 3u) & ~3u;
        if (lane < items4 - items) S.map[items + lane] = 0u, S.val[4 * (items + lane)] = 0.0f;  // pad to whole groups of four
        __syncwarp();
        // Pitch-class fold, lane = class: contributions in (peak, harmonic, offset) order like the reference (extractor.rs:640-664).  An item
        // touches a class at most once, so the lane takes its slot number from the item's map and adds that slot — slot 0 holds 0.0f, and
        // x + 0.0f == x for the non-negative sums here — instead of scanning all 3 x items (class, value) entries.
        if (lane < 12) {
            const int sh = 2 * lane;
            for (uint32_t it = 0; it < items4; it += 4) {
                const uint4 m = *reinterpret_cast<const uint4*>(S.map + it);
                const float* v = S.val + 4 * it;
                pc = pc + v[(m.x >> sh) & 3u];
                pc = pc + v[4 + ((m.y >> sh) & 3u)];
                pc = pc + v[8 + ((m.z >> sh) & 3u)];
                pc = pc + v[12 + ((m.w >> sh) & 3u)];
            }
        }
        // L2 normalise with the reference's sequential sum of squares (extractor.rs:668-677)
        float ss = 0.0f;
        for (int i = 0; i < 12; ++i) {
            const float v = __shfl_sync(0xffffffffu, pc, i);
            ss = ss + v * v;
        }
        const float norm = sqrtf(ss);
        if (norm > 1e-10f) pc = pc / norm;
    }
    __syncwarp();
    return pc;
}

// MAXP peak slots per frame; WARPS frames per CTA (4 x 512 slots or 2 x 2048 slots of shared memory).
// cfg.key_compact: the masked band comes from T.kband (mask_kernel<COMPACT>) and the frame energy from the per-CTA shares in T.kepart.
template <int MAXP, int WARPS, int MAXI = HPCP_MAX_SEL * HPCP_MAX_HARM>
__global__ void __launch_bounds__(32 * WARPS) hpcp_kernel(const TrackDev* __restrict__ tr, const SrTables* __restrict__ srtab, const int32_t* __restrict__ sr_index,
                                                          float* fa, DevCfg cfg) {
    __shared__ HpcpSmem<MAXP, MAXI> sm[WARPS];
    const int t = blockIdx.y;
    const TrackDev& T = tr[t];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t f = blockIdx.x * WARPS + w;
    if (T.status != 0 || f >= T.Fk || T.beat_sync) return;
    HpcpSmem<MAXP, MAXI>& S = sm[w];
    const SrTables& st = srtab[sr_index[t]];
    const uint32_t KBINS = cfg.key_bins;
    // frame energy (extractor.rs:1132-1134).  Consumed only through (E/median)^0.5 frame weights, a
    // tolerance-level quantity, so the 4097-term sum is a tree instead of a serial fold.
    float e = 0.0f;
    const float* row;  // indexed by key-STFT bin
    if (cfg.key_compact) {
        row = fa + T.kband + (uint64_t)f * T.kband_stride - T.kband_lo;
        const uint32_t np = (KBINS + 31) / 32;  // warps of the mask kernel
        for (uint32_t k = lane; k < np; k += 32) e = e + fa[T.kepart + (uint64_t)k * T.kepart_stride + f];
    } else {
        row = fa + T.keyspec + (uint64_t)f * KBINS;
        for (uint32_t k = lane; k < KBINS; k += 32) {
            const float x = row[k];
            e = e + x * x;
        }
    }
    for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
    const float* sel = cfg.key_whiten ? fa + T.kwhite + (uint64_t)f * T.kwhite_stride : row;
    const float res = (float)T.sr / (float)cfg.key_frame;
    const float nyq = (float)T.sr / 2.0f;
    float pc = hpcp_band<MAXP, MAXI>(sel, row, st.key_bin_lo, st.key_bin_hi, fmaxf(100.0f, 20.0f), fminf(5000.0f, nyq), cfg.hpcp_peaks, T.key_tuning, res, S, lane, cfg);
    if (cfg.key_bass_blend) {  // extractor.rs:1154-1239: (1-w) full + w bass, renormalised
        const float bass = hpcp_band<MAXP, MAXI>(sel, row, st.bass_bin_lo, st.bass_bin_hi, st.bass_fmin, st.bass_fmax, min(max(cfg.hpcp_peaks, 1u), 12u), T.key_tuning, res, S,
                                           lane, cfg);
        const float bw = clamp_rs(cfg.bass_weight, 0.0f, 1.0f);
        pc = (1.0f - bw) * pc + bw * bass;
        float ss = 0.0f;
        for (int i = 0; i < 12; ++i) {
            const float v = __shfl_sync(0xffffffffu, pc, i);
            ss = ss + v * v;
        }
        const float norm = sqrtf(ss);
        if (norm > 1e-10f) pc = pc / norm;
    }
    if (lane < 12) fa[T.chroma + (uint64_t)f * 12 + lane] = pc;
    if (lane == 0) fa[T.kenergy + f] = e;
}

// ---- chroma folding (extractor.rs:393-487, enable_key_hpcp = false): one warp per frame ---------------------------
// chroma[pc] = sum over band bins (ascending) of max(x,0)^0.6 * w[bin][pc]; the weights (Gaussian soft mapping in
// circular pitch-class space, or the hard nearest-class assignment) depend only on the bin, so they come from a
// per-sample-rate table grouped by pitch class in the reference's accumulation order.  The 0.6-power of every band bin
// is evaluated once, in parallel, into shared memory; 12 lanes then fold their pitch class.
constexpr int FOLD_MAX = 1024;  // band bins (912 at 44.1 kHz; the ABI rejects sample rates whose band is wider)

// Tracks with a non-zero tuning offset (lib.rs:1098-1121) use per-track lists built by fold_table_kernel (k_keyvar.cu) in the same layout.
// Beat-synchronous tracks (extractor.rs:830-922) fold every frame into chroma2 / kweights, which beat_sync_kernel then averages per beat interval.
__global__ void __launch_bounds__(128) chroma_fold_kernel(const TrackDev* __restrict__ tr, const SrTables* __restrict__ srtab, const int32_t* __restrict__ sr_index,
                                                          float* fa, const int32_t* __restrict__ ia, DevCfg cfg) {
    __shared__ float contrib[4][FOLD_MAX];
    const int t = blockIdx.y;
    const TrackDev& T = tr[t];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t f = blockIdx.x * 4 + w;
    if (T.status != 0 || f >= T.Fk) return;
    if (!T.beat_sync && (cfg.key_hpcp || cfg.key_log_freq)) return;
    const SrTables& st = srtab[sr_index[t]];
    const uint32_t KBINS = cfg.key_bins;
    const float* row = fa + T.keyspec + (uint64_t)f * KBINS;
    float e = 0.0f;  // frame energy: tree sum (tolerance-level consumer, see hpcp_kernel)
    for (uint32_t k = lane; k < KBINS; k += 32) {
        const float x = row[k];
        e = e + x * x;
    }
    for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(0xffffffffu, e, o);
    const uint32_t lo = st.fold_lo, hi = st.fold_hi;
    const bool tuned = cfg.key_tuning && ia[T.kfold_bin + 12 * FOLD_MAX + 12] != 0;
    float pc = 0.0f;
    if (lo <= hi) {
        for (uint32_t b = lo + lane; b <= hi; b += 32) contrib[w][b - lo] = powf(fmaxf(row[b], 0.0f), 0.6f);  // extractor.rs:431
        __syncwarp();
        if (lane < 12) {
            if (tuned) {
                const int32_t* bins = ia + T.kfold_bin + lane * FOLD_MAX;
                const float* ws = fa + T.kfold_w + lane * FOLD_MAX;
                const int n = ia[T.kfold_bin + 12 * FOLD_MAX + lane];
                for (int q = 0; q < n; ++q) pc = pc + contrib[w][bins[q] - lo] * ws[q];
            } else {
                const int a = st.fold_off[lane], z = st.fold_off[lane + 1];
                for (int q = a; q < z; ++q) pc = pc + contrib[w][st.fold_bin[q] - lo] * st.fold_w[q];
            }
        }
        float ss = 0.0f;
        for (int i = 0; i < 12; ++i) {
            const float v = __shfl_sync(0xffffffffu, pc, i);
            ss = ss + v * v;
        }
        const float norm = sqrtf(ss);
        if (norm > 1e-10f) pc = pc / norm;
    }
    if (lane < 12) fa[(T.beat_sync ? T.chroma2 : T.chroma) + (uint64_t)f * 12 + lane] = pc;
    if (lane == 0) fa[(T.beat_sync ? T.kweights : T.kenergy) + f] = e;
}

// ---- sharpen_chroma (chroma/normalization.rs:41-65): thread per frame ----------------------------------------------
__global__ void __launch_bounds__(256) chroma_sharpen_kernel(const TrackDev* __restrict__ tr, float* fa, float power) {
    const TrackDev& T = tr[blockIdx.y];
    const uint32_t f = blockIdx.x * blockDim.x + threadIdx.x;
    if (T.status != 0 || f >= T.kf) return;
    float* ch = fa + T.chroma + (uint64_t)f * 12;
    float v[12], ss = 0.0f;
    for (int i = 0; i < 12; ++i) {
        v[i] = powf(ch[i], power);
        ss = ss + v[i] * v[i];
    }
    const float norm = sqrtf(ss);
    for (int i = 0; i < 12; ++i) ch[i] = norm > 1e-10f ? v[i] / norm : 1.0f / sqrtf(12.0f);
}

// ---- 5-tap median over time per pitch class (smoothing.rs:37-94); applied when Fk > 5 --------------
__global__ void __launch_bounds__(256) chroma_smooth_kernel(const TrackDev* __restrict__ tr, float* fa) {
    const TrackDev& T = tr[blockIdx.y];
    const uint32_t nf = T.kf;
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (T.status != 0 || i >= nf * 12) return;
    const float* src = fa + T.chroma;
    float* dst = fa + T.chroma2;
    if (nf <= 5) {
        dst[i] = src[i];
        return;
    }
    const int t = (int)(i / 12), s = (int)(i % 12);
    float v[5];
    int n = 0;
    for (int off = -2; off <= 2; ++off) {
        const int ft = t + off;
        if (ft >= 0 && ft < (int)nf) v[n++] = src[(uint64_t)ft * 12 + s];
    }
    for (int a = 1; a < n; ++a) {  // insertion sort; equal keys are indistinguishable
        const float x = v[a];
        int j = a;
        while (j > 0 && v[j - 1] > x) {
            v[j] = v[j - 1];
            --j;
        }
        v[j] = x;
    }
    dst[i] = v[n / 2];
}

// ---- frame weights (lib.rs:1236-1287): one CTA per track -------------------------------------------
// Works on the (optionally edge-trimmed, lib.rs:1216-1233) slice [f0, f0 + nf) of the smoothed chroma; weights are
// stored at slice-relative indices.
__global__ void __launch_bounds__(256) key_weights_kernel(TrackDev* tr, float* fa, DevCfg cfg) {
    __shared__ uint32_t hist[256];
    __shared__ uint32_t bc[2];
    __shared__ float sred[32];
    __shared__ uint32_t sused[32];
    TrackDev& T = tr[blockIdx.x];
    uint32_t f0, nf;
    key_slice(T.kf, cfg, &f0, &nf);
    if (threadIdx.x == 0) T.have_w = 0;
    if (T.status != 0 || nf == 0 || !cfg.key_weighting) return;
    const float* en = fa + T.kenergy + f0;
    const float median = fmaxf(block_select_kth(en, nf, nf / 2, hist, bc), 1e-12f);
    const float* ch = fa + T.chroma2 + (uint64_t)f0 * 12;
    float* wv = fa + T.kweights;
    const float tp = fmaxf(cfg.key_tonal_pow, 0.0f), ep = fmaxf(cfg.key_energy_pow, 0.0f);
    const float ln12 = logf(12.0f);
    float sw = 0.0f;
    uint32_t used = 0;
    for (uint32_t t = threadIdx.x; t < nf; t += blockDim.x) {
        const float* c = ch + (uint64_t)t * 12;
        float sum = 0.0f;
        for (int i = 0; i < 12; ++i) sum = sum + c[i];
        float tonal = 0.0f;
        if (sum > 1e-12f) {
            float ent = 0.0f;
            for (int i = 0; i < 12; ++i) {
                const float p = c[i] / sum;
                if (p > 1e-12f) ent = ent - p * logf(p);
            }
            tonal = clamp_rs(1.0f - (ent / ln12), 0.0f, 1.0f);
        }
        if (tonal < cfg.key_min_tonal) tonal = 0.0f;
        const float e = fmaxf(en[t] / median, 0.0f);
        const float wt = (tp == 2.0f) ? tonal * tonal : powf(tonal, tp);
        const float we = (ep == 0.5f) ? sqrtf(e) : powf(e, ep);
        const float wgt = fmaxf(wt * we, 0.0f);
        wv[t] = wgt;
        sw += wgt;
        used += wgt > 0.0f;
    }
    for (int o = 16; o > 0; o >>= 1) {
        sw += __shfl_xor_sync(0xffffffffu, sw, o);
        used += __shfl_xor_sync(0xffffffffu, used, o);
    }
    if ((threadIdx.x & 31) == 0) {
        sred[threadIdx.x >> 5] = sw;
        sused[threadIdx.x >> 5] = used;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        float s = 0.0f;
        uint32_t u = 0;
        for (int q = 0; q < (int)(blockDim.x >> 5); ++q) {
            s += sred[q];
            u += sused[q];
        }
        T.have_w = !(s <= 1e-12f || u < 10) ? 1 : 0;
    }
}

// Rows a launch covers: the first pass scores every window row (and both whole-track rows of the ensemble); the
// whole-track row of a voting / multi-scale track is only needed when no window passes the clarity gate
// (lib.rs:1385-1411, detector.rs:648-668), so it is computed by a second pass (fallback_only) for the tracks
// key_vote_kernel flagged.  Returns false when this (track, row, pass) has nothing to do.
__device__ __forceinline__ bool key_row_for_pass(const TrackDev& T, const DevCfg& cfg, uint32_t bx, int fallback_only, uint32_t* f0, uint32_t* nf, KeyRows* R,
                                                 uint32_t* row) {
    if (T.status != 0 || T.kf == 0) return false;
    key_slice(T.kf, cfg, f0, nf);
    if (*nf == 0) return false;
    *R = key_rows(*nf, cfg);
    if (R->mode == KEY_ROWS_ENSEMBLE) {
        *row = bx;
        return !fallback_only && bx < 2 && bx < T.seg_cap;
    }
    if (fallback_only) {
        *row = R->nseg;
        return bx == 0 && T.key_fallback && *row < T.seg_cap;
    }
    *row = bx;
    if (R->nseg == 0) return bx == 0;  // no windows: the whole-track row is the result
    return bx < R->nseg && bx < T.seg_cap;
}

// ---- template scores: one warp per (row, key) -----------------------------------------------------------
// score = sum over frames (in frame order) of w_t * <c_t, T_k> (detector.rs:984-1001).  The 32 lanes
// evaluate the 12-term dot products of 32 consecutive frames in parallel (each in the reference's term
// order); the running sum then absorbs the 32 products strictly in frame order through shuffles, so the
// result equals the serial fold bit for bit while the chain per frame is one add instead of ~25 ops.
// blockIdx.x = row (key_rows.cuh); blockDim = 24 warps, warp = key.
__global__ void __launch_bounds__(768) segment_score_kernel(const TrackDev* __restrict__ tr, float* fa, Tables tab, DevCfg cfg, int fallback_only) {
    const TrackDev& T = tr[blockIdx.y];
    uint32_t f0, nf, row;
    KeyRows R;
    if (!key_row_for_pass(T, cfg, blockIdx.x, fallback_only, &f0, &nf, &R, &row)) return;
    uint32_t start, len;
    float scale_w;
    int tset;
    key_row_range(R, row, nf, cfg, &start, &len, &scale_w, &tset);
    const int k = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* tmaj = tset == 1 ? tab.key_major_tp : tab.key_major;
    const float* tmin = tset == 1 ? tab.key_minor_tp : tab.key_minor;
    const float* tpl = (k < 12 ? tmaj + k * 12 : tmin + (k - 12) * 12);
    float tp[12];
#pragma unroll
    for (int i = 0; i < 12; ++i) tp[i] = tpl[i];
    const float* ch = fa + T.chroma2 + (uint64_t)(f0 + start) * 12;
    const float* wv = T.have_w ? fa + T.kweights + start : nullptr;
    float acc = 0.0f;
    for (uint32_t t0 = 0; t0 < len; t0 += 32) {
        const uint32_t t = t0 + lane;
        float prod = 0.0f;
        bool use = false;
        if (t < len) {
            const float* c = ch + (uint64_t)t * 12;
            float dot = 0.0f;
#pragma unroll
            for (int i = 0; i < 12; ++i) dot = dot + c[i] * tp[i];
            if (wv) {
                const float wt = wv[t];
                use = wt > 0.0f;
                prod = wt * dot;
            } else {
                use = true;
                prod = dot;
            }
        }
        const uint32_t um = __ballot_sync(0xffffffffu, use);
#pragma unroll
        for (int l = 0; l < 32; ++l) {
            const float p = __shfl_sync(0xffffffffu, prod, l);
            if ((um >> l) & 1u) acc = acc + p;
        }
    }
    if (lane == 0) fa[T.seg_scores + (uint64_t)row * 24 + k] = acc;
}

// ---- weighted chroma sums of a row (mode heuristic, detector.rs:345-371): warp i < 12 folds avg[i] += w_t * c_t[i] over the
// frames with w_t > 0 in frame order (or avg[i] += c_t[i] without weights); warp 12 folds the weight sum.  Same
// "parallel products, ordered absorption" scheme as the score kernel.  blockDim = 13 warps.
__global__ void __launch_bounds__(416) segment_avg_kernel(const TrackDev* __restrict__ tr, float* fa, DevCfg cfg, int fallback_only) {
    const TrackDev& T = tr[blockIdx.y];
    uint32_t f0, nf, row;
    KeyRows R;
    if (!key_row_for_pass(T, cfg, blockIdx.x, fallback_only, &f0, &nf, &R, &row)) return;
    uint32_t start, len;
    float scale_w;
    int tset;
    key_row_range(R, row, nf, cfg, &start, &len, &scale_w, &tset);
    const int i = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* ch = fa + T.chroma2 + (uint64_t)(f0 + start) * 12;
    const float* wv = T.have_w ? fa + T.kweights + start : nullptr;
    float acc = 0.0f;
    if (!wv && i == 12) {
        acc = (float)len;  // wsum = chroma_vectors.len() as f32
    } else {
        for (uint32_t t0 = 0; t0 < len; t0 += 32) {
            const uint32_t t = t0 + lane;
            float prod = 0.0f;
            bool use = false;
            if (t < len) {
                const float c = i < 12 ? ch[(uint64_t)t * 12 + i] : 1.0f;
                if (wv) {
                    const float wt = wv[t];
                    use = wt > 0.0f;
                    prod = i < 12 ? wt * c : wt;
                } else {
                    use = true;
                    prod = c;
                }
            }
            const uint32_t um = __ballot_sync(0xffffffffu, use);
#pragma unroll
            for (int l = 0; l < 32; ++l) {
                const float p = __shfl_sync(0xffffffffu, prod, l);
                if ((um >> l) & 1u) acc = acc + p;
            }
        }
    }
    if (lane == 0) fa[T.seg_avg + (uint64_t)row * 13 + i] = acc;
}

// detect_key_weighted steps 1.5 - 2 on 24 raw scores: ranked keys/scores out (detector.rs:135-250) and the
// same refined scores indexed by key id (by_key).  Kept out of line: each call gets its own stack
// frame, so the caller's accumulators never share local-memory slots with this function's temporaries.
__device__ __noinline__ void rank_keys(const float* raw, int* keys, float* scores, float* by_key) {
    float sc[24];
    for (int k = 0; k < 24; ++k) sc[k] = raw[k];
    float mxM = 0.0f, mxm = 0.0f;
    for (int k = 0; k < 12; ++k) mxM = fmaxf(mxM, sc[k]);
    for (int k = 12; k < 24; ++k) mxm = fmaxf(mxm, sc[k]);
    if (mxM > 1e-9f && mxm > 1e-9f) {
        for (int k = 0; k < 12; ++k) sc[k] = sc[k] / mxM;
        for (int k = 12; k < 24; ++k) sc[k] = sc[k] / mxm;
    }
    const int pos_of[12] = {0, 7, 2, 9, 4, 11, 6, 1, 8, 3, 10, 5};  // position of tonic on the circle of fifths (self-inverse table)
    int topM = 0, topm = 12;
    for (int k = 0; k < 12; ++k)
        if (sc[k] >= sc[topM]) topM = k;  // max_by: last maximal
    for (int k = 12; k < 24; ++k)
        if (sc[k] >= sc[topm]) topm = k;
    float refined[24];
    for (int k = 0; k < 24; ++k) {
        refined[k] = sc[k];
        const int ref = k < 12 ? topM : topm;
        const float ref_score = sc[ref];
        if (ref_score > 1e-9f) {
            const int d = abs(pos_of[k % 12] - pos_of[ref % 12]);
            const int dist = min(d, 12 - d);
            if (dist <= 2) {
                const float bonus = 0.20f * (1.0f - (float)dist * 0.5f);
                refined[k] = refined[k] + ref_score * bonus;
            }
        }
    }
    for (int k = 0; k < 24; ++k) by_key[k] = refined[k];
    for (int k = 0; k < 24; ++k) {  // stable insertion sort, descending
        const float x = refined[k];
        int j = k;
        while (j > 0 && scores[j - 1] < x) {
            scores[j] = scores[j - 1];
            keys[j] = keys[j - 1];
            --j;
        }
        scores[j] = x;
        keys[j] = k;
    }
}

__device__ __noinline__ float key_clarity(const float* sc, int n) {  // key_clarity.rs:51-93
    if (n < 2) return 0.0f;
    float sum = 0.0f;
    for (int i = 0; i < n; ++i) sum = sum + sc[i];
    const float avg = sum / (float)n;
    float mn = sc[0], mx = sc[0];
    for (int i = 1; i < n; ++i) {
        if (sc[i] < mn) mn = sc[i];
        if (sc[i] >= mx) mx = sc[i];
    }
    const float range = mx - mn;
    if (range > 1e-10f) return clamp_rs((sc[0] - avg) / range, 0.0f, 1.0f);
    return 0.0f;
}

// Stable descending sort of 24 (key, score) pairs already in some order (Rust sort_by is stable).
__device__ __forceinline__ void stable_sort_desc(int* keys, float* scores) {
    for (int a = 1; a < 24; ++a) {
        const float x = scores[a];
        const int kx = keys[a];
        int j = a;
        while (j > 0 && scores[j - 1] < x) {
            scores[j] = scores[j - 1];
            keys[j] = keys[j - 1];
            --j;
        }
        scores[j] = x;
        keys[j] = kx;
    }
}

// detect_key_weighted_mode_heuristic after the base scoring (detector.rs:338-517): minor-key leading-tone bonus, stable
// re-sort, scale-degree mode preference, optional parallel-mode flip.  keys/scores (ranked) and by_key are updated in
// place; returns the chosen key and its confidence.
__device__ __noinline__ void mode_heuristic(const float* avg13, const DevCfg& cfg, int* keys, float* scores, float* by_key, int* chosen_out, float* conf_out) {
    const float flip_ratio = clamp_rs(cfg.key_flip_ratio, 0.0f, 1.0f);
    const bool enable_flip = flip_ratio > 0.0f;
    const float wsum = avg13[12];
    if ((!cfg.key_minor_bonus && !enable_flip) || wsum <= 1e-9f) return;  // base result stands
    float avg[12];
    float sum = 0.0f;
    for (int i = 0; i < 12; ++i) {
        avg[i] = avg13[i];
        sum = sum + avg[i];
    }
    if (sum > 1e-9f)
        for (int i = 0; i < 12; ++i) avg[i] = avg[i] / sum;
    if (cfg.key_minor_bonus) {
        const float bw = fmaxf(cfg.key_minor_bonus_w, 0.0f);
        if (bw > 0.0f)
            for (int i = 0; i < 24; ++i)
                if (keys[i] >= 12) {
                    const int tonic = keys[i] - 12;
                    scores[i] = scores[i] + wsum * bw * (avg[(tonic + 11) % 12] - avg[(tonic + 10) % 12]);
                }
    }
    stable_sort_desc(keys, scores);
    for (int i = 0; i < 24; ++i) by_key[keys[i]] = scores[i];
    const int best_key = keys[0];
    const int tonic = best_key % 12;
    const bool best_is_major = best_key < 12;
    const float p_min3 = avg[(tonic + 3) % 12], p_maj3 = avg[(tonic + 4) % 12];
    const float p_min6 = avg[(tonic + 8) % 12], p_maj6 = avg[(tonic + 9) % 12];
    const float p_min7 = avg[(tonic + 10) % 12], p_maj7 = avg[(tonic + 11) % 12];
    const float margin = fmaxf(cfg.key_third_margin, 0.0f);
    float minor_score = 0.0f, major_score = 0.0f;
    const float d3 = fabsf(p_min3 - p_maj3);
    if (p_min3 > (p_maj3 * (1.0f + margin))) minor_score = minor_score + d3 * 2.0f;
    else if (p_maj3 > (p_min3 * (1.0f + margin))) major_score = major_score + d3 * 2.0f;
    const float d6 = fabsf(p_min6 - p_maj6);
    if (p_min6 > (p_maj6 * (1.0f + margin))) minor_score = minor_score + d6 * 1.0f;
    else if (p_maj6 > (p_min6 * (1.0f + margin))) major_score = major_score + d6 * 1.0f;
    const float d7 = fabsf(p_min7 - p_maj7);
    if (p_min7 > (p_maj7 * (1.0f + margin))) minor_score = minor_score + d7 * 1.0f;
    else if (p_maj7 > (p_min7 * (1.0f + margin))) major_score = major_score + d7 * 1.0f;
    const float total = minor_score + major_score;
    const bool minor_pref = total > 1e-9f ? minor_score > major_score * (1.0f + margin * 0.5f) : false;
    const bool major_pref = total > 1e-9f ? major_score > minor_score * (1.0f + margin * 0.5f) : false;
    int chosen = best_key;
    if (enable_flip) {
        if (best_is_major && minor_pref) {
            const float s_best = by_key[tonic], s_alt = by_key[12 + tonic];
            if (s_best > 0.0f && s_alt >= s_best * flip_ratio) chosen = 12 + tonic;
        } else if (!best_is_major && major_pref) {
            const float s_best = by_key[12 + tonic], s_alt = by_key[tonic];
            if (s_best > 0.0f && s_alt >= s_best * flip_ratio) chosen = tonic;
        }
    }
    const float chosen_score = by_key[chosen];
    float best_other = 0.0f;
    for (int i = 0; i < 24; ++i)
        if (keys[i] != chosen) best_other = fmaxf(best_other, scores[i]);
    *chosen_out = chosen;
    *conf_out = chosen_score > 0.0f ? clamp_rs((chosen_score - best_other) / chosen_score, 0.0f, 1.0f) : 0.0f;
}

// ---- per-row detection result: one thread per (row, track) ----------------------------------------------------------------
// seg_rank[row] = { refined score by key id [24], clarity of the ranked table, chosen key, confidence, 0 }
__global__ void __launch_bounds__(64) row_rank_kernel(const TrackDev* __restrict__ tr, float* fa, DevCfg cfg, uint32_t max_rows, int fallback_only) {
    const TrackDev& T = tr[blockIdx.y];
    const uint32_t bx = blockIdx.x * blockDim.x + threadIdx.x;
    if (bx >= max_rows) return;
    uint32_t f0, nf, row;
    KeyRows R;
    if (!key_row_for_pass(T, cfg, bx, fallback_only, &f0, &nf, &R, &row)) return;
    int keys[24];
    float scores[24], by_key[24];
    rank_keys(fa + T.seg_scores + (uint64_t)row * 24, keys, scores, by_key);
    // weighted top-3 vote (detector.rs:254-275): three distinct keys, so the first-ranked key wins
    int chosen = keys[0];
    float conf = scores[0] > 0.0f ? clamp_rs((scores[0] - scores[1]) / scores[0], 0.0f, 1.0f) : 0.0f;
    if (cfg.key_heur && R.mode != KEY_ROWS_ENSEMBLE) mode_heuristic(fa + T.seg_avg + (uint64_t)row * 13, cfg, keys, scores, by_key, &chosen, &conf);
    float* out = fa + T.seg_rank + (uint64_t)row * 28;
    for (int k = 0; k < 24; ++k) out[k] = by_key[k];
    out[24] = key_clarity(scores, 24);
    out[25] = (float)chosen;
    out[26] = conf;
    out[27] = 0.0f;
}

// Sort 24 accumulated scores (by key id) descending, stable in key-id order; confidence as lib.rs:1412-1425.
__device__ __forceinline__ void finish_accumulated(const float* acc, int* keys, float* fin, int* key, float* confidence) {
    for (int k = 0; k < 24; ++k) {
        const float x = acc[k];
        int j = k;
        while (j > 0 && fin[j - 1] < x) {
            fin[j] = fin[j - 1];
            keys[j] = keys[j - 1];
            --j;
        }
        fin[j] = x;
        keys[j] = k;
    }
    *key = keys[0];
    *confidence = fin[0] > 0.0f ? clamp_rs((fin[0] - fin[1]) / fin[0], 0.0f, 1.0f) : 0.0f;
}

// ---- per-track decision (lib.rs:1290-1461): one thread per track ---------------------------------------------------------
__global__ void key_vote_kernel(TrackDev* tr, const float* fa, int n_tracks, DevCfg cfg, int fallback_only) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tracks) return;
    TrackDev& T = tr[t];
    if (fallback_only) {
        if (!T.key_fallback) return;
    } else {
        T.key = 0;
        T.key_confidence = 0.0f;
        T.key_clarity = 0.0f;
        T.key_fallback = 0;
    }
    if (T.status != 0 || T.kf == 0 || T.m < cfg.frame) return;  // so_key.cpp:790: shorter than frame_size
    uint32_t f0, nf;
    key_slice(T.kf, cfg, &f0, &nf);
    if (nf == 0) return;
    const KeyRows R = key_rows(nf, cfg);
    const float* rk = fa + T.seg_rank;
    int keys[24];
    float fin[24];
    int key = 0;
    float confidence = 0.0f;
    if (R.mode == KEY_ROWS_ENSEMBLE) {  // detector.rs:881-976
        const float total = cfg.key_ens_kk + cfg.key_ens_tp;
        const float kk_norm = total > 1e-9f ? cfg.key_ens_kk / total : 0.5f;
        const float tp_norm = total > 1e-9f ? cfg.key_ens_tp / total : 0.5f;
        float comb[24];
        for (int k = 0; k < 24; ++k) comb[k] = kk_norm * rk[k] + tp_norm * rk[28 + k];
        finish_accumulated(comb, keys, fin, &key, &confidence);
        T.key = key;
        T.key_confidence = confidence;
        T.key_clarity = key_clarity(fin, 24);
        return;
    }
    const uint32_t nseg = min(R.nseg, T.seg_cap > 0 ? T.seg_cap - 1 : 0u);
    if (nseg > 0 && !fallback_only) {
        const bool ms = R.mode == KEY_ROWS_MULTI_SCALE;
        const float min_cl = clamp_rs(ms ? cfg.ms_min_clarity : cfg.key_seg_min_clarity, 0.0f, 1.0f);
        float acc[24];
        for (int k = 0; k < 24; ++k) acc[k] = 0.0f;
        uint32_t used = 0;
        float total_weight = 0.0f;
        for (uint32_t s = 0; s < nseg; ++s) {
            const float* r = rk + (uint64_t)s * 28;
            const float cl = r[24];
            if (cl >= min_cl) {
                ++used;
                float cw = cl;
                if (ms) {  // detector.rs:634-645: clarity x scale weight
                    uint32_t start, len;
                    float scale_w;
                    int tset;
                    key_row_range(R, s, nf, cfg, &start, &len, &scale_w, &tset);
                    cw = cl * scale_w;
                    total_weight = total_weight + cw;
                }
                for (int k = 0; k < 24; ++k) acc[k] = acc[k] + r[k] * cw;  // one add per key and row, as lib.rs:1375-1381
            }
        }
        const bool ok = ms ? (used > 0 && !(total_weight <= 1e-12f)) : used > 0;
        if (!ok) {
            T.key_fallback = 1;  // every window rejected: the whole-track row is computed on demand
            return;
        }
        if (ms)
            for (int k = 0; k < 24; ++k) acc[k] = acc[k] / total_weight;
        finish_accumulated(acc, keys, fin, &key, &confidence);
        T.key = key;
        T.key_confidence = confidence;
        T.key_clarity = key_clarity(fin, 24);
        return;
    }
    // whole-track detection: the row's own result; its ranked table gives the clarity (lib.rs:1461)
    const float* r = rk + (uint64_t)nseg * 28;
    T.key = (int)r[25];
    T.key_confidence = r[26];
    T.key_clarity = r[24];
}

void launch_key_mask(const WaveCtx& c) {
    if (c.max_Fk > 0 && !c.cfg.key_hpss && (c.cfg.key_mask || c.cfg.key_smooth_only)) {  // the median-HPSS mask takes precedence (lib.rs:1011-1030)
        dim3 g((c.cfg.key_bins + 127) / 128, c.n_tracks);
        const bool fast = !c.cfg.key_smooth_only && fmaxf(c.cfg.key_mask_power, 1.0f) == 2.0f && c.cfg.key_bins == 4097;
        // Few long tracks: cut the time axis so that the launch has about four CTAs per SM (see mask_kernel); segments of at least 2048
        // frames, at most MASK_SEG_MAX per track (the prefix rows planned in engine.cu).
        uint32_t seg_len = 0;
        if (c.cfg.key_compact && c.cfg.key_margin == 12 && fast && c.max_Fk >= 8192 && g.x * g.y < 300) {
            const uint32_t want = std::min<uint32_t>(MASK_SEG_MAX, 592u / (g.x * g.y));
            seg_len = std::max<uint32_t>(2048u, ((c.max_Fk / std::max(want, 1u)) + 31u) & ~31u);
            const uint32_t nseg = std::max(1u, c.max_Fk / seg_len);
            if (nseg < 2) seg_len = 0;
            else {
                g.z = nseg;
                mask_prefix_kernel<4097><<<dim3(g.x, g.y), 128, 0, c.stream>>>(c.tracks, c.fa, c.cfg, seg_len);
                count_launch("key_mask");
            }
        }
        if (c.cfg.key_compact) {
            if (c.cfg.key_margin == 12 && fast && c.kband_stride_common == 960) mask_kernel<12, true, 4097, true, 960><<<g, 128, 0, c.stream>>>(c.tracks, c.fa, c.cfg, seg_len);  // defaults (config.rs:669, 680, 688) at >= 39.2 kHz
            else if (c.cfg.key_margin == 12 && fast) mask_kernel<12, true, 4097, true><<<g, 128, 0, c.stream>>>(c.tracks, c.fa, c.cfg, seg_len);
            else if (c.cfg.key_margin == 12) mask_kernel<12, false, 0, true><<<g, 128, 0, c.stream>>>(c.tracks, c.fa, c.cfg, 0u);
            else mask_kernel<0, false, 0, true><<<g, 128, 0, c.stream>>>(c.tracks, c.fa, c.cfg, 0u);
        } else {
            if (c.cfg.key_margin == 12 && fast) mask_kernel<12, true, 4097, false><<<g, 128, 0, c.stream>>>(c.tracks, c.fa, c.cfg, 0u);
            else if (c.cfg.key_margin == 12) mask_kernel<12, false, 0, false><<<g, 128, 0, c.stream>>>(c.tracks, c.fa, c.cfg, 0u);
            else mask_kernel<0, false, 0, false><<<g, 128, 0, c.stream>>>(c.tracks, c.fa, c.cfg, 0u);
        }
        count_launch("key_mask");
    }
    if (c.max_Fk > 0) launch_key_variants_pre(c);
}

void launch_key_hpcp(const WaveCtx& c) {
    if (c.max_Fk > 0) {
        const dim3 g((c.max_Fk + 3) / 4, c.n_tracks);
        // HPCP peak slots: 512 cover the 100..5000 Hz band down to 39.2 kHz; lower sample rates put more key-STFT bins into the band
        // which chroma front end a track takes is decided per track (lib.rs:1123-1197): beat-synchronous tracks and plain chroma
        // folding go through chroma_fold_kernel, log-frequency through k_keyvar.cu, everything else through HPCP
        if (c.cfg.key_hpcp && !c.cfg.key_log_freq) {
            const uint32_t max_items = std::min(std::max(c.cfg.hpcp_peaks, 1u), (uint32_t)HPCP_MAX_SEL) * std::min(std::max(c.cfg.hpcp_harm, 1u), (uint32_t)HPCP_MAX_HARM);
            if (c.max_key_peaks <= (uint32_t)HPCP_PEAKS_44K && max_items <= 128) hpcp_kernel<HPCP_PEAKS_44K, 4, 128><<<g, 128, 0, c.stream>>>(c.tracks, c.srtab, c.sr_index, c.fa, c.cfg);
            else if (c.max_key_peaks <= (uint32_t)HPCP_PEAKS_44K) hpcp_kernel<HPCP_PEAKS_44K, 4><<<g, 128, 0, c.stream>>>(c.tracks, c.srtab, c.sr_index, c.fa, c.cfg);
            else hpcp_kernel<HPCP_PEAKS_ANY, 2><<<dim3((c.max_Fk + 1) / 2, c.n_tracks), 64, 0, c.stream>>>(c.tracks, c.srtab, c.sr_index, c.fa, c.cfg);
            count_launch("key_hpcp");
        }
        if (c.cfg.key_beat_sync || (!c.cfg.key_hpcp && !c.cfg.key_log_freq)) {
            chroma_fold_kernel<<<g, 128, 0, c.stream>>>(c.tracks, c.srtab, c.sr_index, c.fa, c.ia, c.cfg);
            count_launch("key_hpcp");
        }
        launch_key_chroma_variants(c);
        if (c.cfg.chroma_sharpen > 1.0f) {  // lib.rs:1200-1208
            chroma_sharpen_kernel<<<dim3((c.max_Fk + 255) / 256, c.n_tracks), 256, 0, c.stream>>>(c.tracks, c.fa, c.cfg.chroma_sharpen);
            count_launch("key_hpcp");
        }
    }
}

void launch_key_vote(const WaveCtx& c) {
    const uint32_t rows = c.max_seg_cap;
    auto pass = [&](int fallback_only) {
        const uint32_t gx = fallback_only ? 1u : rows;
        segment_score_kernel<<<dim3(gx, c.n_tracks), 768, 0, c.stream>>>(c.tracks, c.fa, c.tab, c.cfg, fallback_only);
        count_launch("key_vote");
        if (c.cfg.key_heur && c.cfg.key_mode != KEY_ROWS_ENSEMBLE) {
            segment_avg_kernel<<<dim3(gx, c.n_tracks), 416, 0, c.stream>>>(c.tracks, c.fa, c.cfg, fallback_only);
            count_launch("key_vote");
        }
        row_rank_kernel<<<dim3((gx + 63) / 64, c.n_tracks), 64, 0, c.stream>>>(c.tracks, c.fa, c.cfg, gx, fallback_only);
        count_launch("key_vote");
    };
    if (c.max_Fk > 0) {
        chroma_smooth_kernel<<<dim3((c.max_Fk * 12 + 255) / 256, c.n_tracks), 256, 0, c.stream>>>(c.tracks, c.fa);
        count_launch("key_vote");
        key_weights_kernel<<<c.n_tracks, 256, 0, c.stream>>>(c.tracks, c.fa, c.cfg);
        count_launch("key_vote");
        pass(0);
    }
    key_vote_kernel<<<(c.n_tracks + 63) / 64, 64, 0, c.stream>>>(c.tracks, c.fa, c.n_tracks, c.cfg, 0);
    count_launch("key_vote");
    if (c.max_Fk > 0 && c.cfg.key_mode != KEY_ROWS_ENSEMBLE && (c.cfg.key_voting || c.cfg.key_mode == KEY_ROWS_MULTI_SCALE)) {
        // rare path: tracks whose windows were all rejected
        pass(1);
        key_vote_kernel<<<(c.n_tracks + 63) / 64, 64, 0, c.stream>>>(c.tracks, c.fa, c.n_tracks, c.cfg, 1);
        count_launch("key_vote");
    }
}

}  // namespace sb
