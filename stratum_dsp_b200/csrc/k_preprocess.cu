// Preprocessing kernels: peak normalisation gain (reference preprocessing/normalization.rs:262-322)
// and silence detection + trim (preprocessing/silence.rs:102-279).
//
// Data layout: tracks are concatenated in one f32 buffer; the gain is never written back — every
// consumer multiplies on load with one rounding (`x*g`), which is bit-identical to the reference's
// in-place `*sample *= gain` followed by a read.
#include "framed.cuh"
#include "kernels.h"

namespace sb {

// ---- peak: order-free exact max|x| per track ------------------------------------------------
__global__ void __launch_bounds__(256) peak_kernel(const float* __restrict__ x, TrackDev* tr) {
    const int t = blockIdx.y;
    const uint64_t n = tr[t].n;
    const float* p = x + tr[t].off;
    float m = 0.0f;
    // float4 body when the track start is 16-byte aligned, scalar otherwise
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if ((((uintptr_t)p) & 15) == 0) {
        const float4* p4 = reinterpret_cast<const float4*>(p);
        const uint64_t n4 = n >> 2;
        for (uint64_t j = i; j < n4; j += stride) {
            float4 v = __ldg(p4 + j);
            m = fmaxf(m, fmaxf(fmaxf(fabsf(v.x), fabsf(v.y)), fmaxf(fabsf(v.z), fabsf(v.w))));
        }
        for (uint64_t j = (n4 << 2) + i; j < n; j += stride) m = fmaxf(m, fabsf(p[j]));
    } else {
        for (uint64_t j = i; j < n; j += stride) m = fmaxf(m, fabsf(p[j]));
    }
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    __shared__ float sm[8];
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < 32) {
        m = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : 0.0f;
        for (int o = 4; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
        if (threadIdx.x == 0) atomicMax(reinterpret_cast<unsigned int*>(&tr[t].peak), __float_as_uint(m));  // m >= 0: bit order == value order
    }
}

// normalize_peak (normalization.rs:275-295) / normalize_rms (:325-398).  Loudness gains are computed on the host
// from the device's block energies (log10f / powf of the host libm, see engine.cu) and passed in `lufs_gain`.
__global__ void gain_kernel(TrackDev* tr, int n_tracks, DevCfg cfg, const float* __restrict__ lufs_gain) {
    int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_tracks) return;
    float g = 1.0f;
    if (cfg.enable_normalization && tr[t].status == 0) {
        const float peak = tr[t].peak;
        if (cfg.normalization == STRATUM_NORM_PEAK) {
            if (peak > 1e-10f) {
                g = cfg.target_peak / peak;
                g = fminf(g, 1.0f / peak);
            }
        } else if (cfg.normalization == STRATUM_NORM_RMS) {
            const float rms = sqrtf(tr[t].rms_sum / (float)tr[t].n);
            if (rms > 1e-10f) {
                g = cfg.rms_target / rms;
                if (peak * g > 1.0f) g = 1.0f / peak;  // :362-379
            }
        } else if (lufs_gain) {
            g = lufs_gain[t];
        }
    }
    tr[t].gain = g;
}

// ---- RMS: the reference folds x*x left to right in f32 over the whole track (normalization.rs:337-343) ----
// One warp per track: 32 coalesced samples per step, every lane then adds the 32 squares in sample order
// (shuffle broadcast), so the sum equals the serial fold bit for bit; the add chain is the critical path.
__global__ void __launch_bounds__(32) rms_seq_kernel(const float* __restrict__ x, TrackDev* tr) {
    TrackDev& T = tr[blockIdx.x];
    if (T.status != 0) return;
    const int lane = threadIdx.x;
    const float* p = x + T.off;
    const uint64_t n = T.n;
    float sum = 0.0f;
    for (uint64_t base = 0; base < n; base += 32) {
        const float v = base + lane < n ? p[base + lane] : 0.0f;
        const float sq = __fmul_rn(v, v);
#pragma unroll
        for (int l = 0; l < 32; ++l) sum = __fadd_rn(sum, __shfl_sync(0xffffffffu, sq, l));  // tail lanes add +0.0
    }
    if (lane == 0) T.rms_sum = sum;
}

// ---- LUFS (normalization.rs:112-259): K-weighting biquad + 400 ms block mean squares ----------------------
// The biquad (DF-II-T) is a linear recurrence  s' = A s + B x.  It is evaluated block-parallel: the track is cut
// into the reference's own 400 ms blocks, (1) every block is run from a zero state to get its end state z_c,
// (2) the block start states follow from the affine scan  s_{c+1} = P s_c + z_c  (P = A^len, composed as 2x2
// affine maps with warp shuffles), (3) every block is re-run from its true start state and its squares are
// summed in sample order.  One lane per block; a warp transposes 32x32 sample tiles through shared memory so
// global loads stay coalesced.
struct Biquad {
    float b0, b1, b2, a1, a2;
};
__device__ __forceinline__ float biquad_step(const Biquad& q, float s, float& x1, float& x2) {  // :161-167
    const float out = __fadd_rn(__fmul_rn(q.b0, s), x1);
    x1 = __fsub_rn(__fadd_rn(__fmul_rn(q.b1, s), x2), __fmul_rn(q.a1, out));
    x2 = __fsub_rn(__fmul_rn(q.b2, s), __fmul_rn(q.a2, out));
    return out;
}

template <bool ENERGY>
__global__ void __launch_bounds__(128) lufs_block_kernel(const float* __restrict__ x, const TrackDev* __restrict__ tr, const SrTables* __restrict__ srtab,
                                                         const int32_t* __restrict__ sr_index, float* fa) {
    __shared__ float tiles[4][32][33];
    const int t = blockIdx.y;
    const TrackDev& T = tr[t];
    if (T.status != 0) return;
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t nb = T.lufs_nb, B = T.lufs_block;
    const uint32_t blk0 = (blockIdx.x * 4 + w) * 32;
    if (blk0 >= nb) return;
    const SrTables& st = srtab[sr_index[t]];
    const Biquad q{st.kw_b0, st.kw_b1, st.kw_b2, st.kw_a1, st.kw_a2};
    float(*tile)[33] = tiles[w];
    const float* p = x + T.off;
    const uint64_t n = T.n;
    const uint32_t blk = blk0 + lane;
    const uint64_t my_start = (uint64_t)blk * B;
    const uint32_t my_len = blk < nb ? (uint32_t)min((uint64_t)B, n - my_start) : 0;
    float x1 = 0.0f, x2 = 0.0f, sum = 0.0f;
    if (ENERGY && blk < nb) {
        x1 = fa[T.lufs_s + 2 * (uint64_t)blk];
        x2 = fa[T.lufs_s + 2 * (uint64_t)blk + 1];
    }
    for (uint32_t jb = 0; jb < B; jb += 32) {
#pragma unroll 4
        for (int r = 0; r < 32; ++r) {
            const uint64_t idx = (uint64_t)(blk0 + r) * B + jb + lane;
            tile[r][lane] = (blk0 + r < nb && jb + lane < B && idx < n) ? p[idx] : 0.0f;
        }
        __syncwarp();
        const uint32_t lim = my_len > jb ? min(my_len - jb, 32u) : 0u;
        for (uint32_t j = 0; j < lim; ++j) {
            const float out = biquad_step(q, tile[lane][j], x1, x2);
            if (ENERGY) sum = __fadd_rn(sum, __fmul_rn(out, out));  // :218
        }
        __syncwarp();
    }
    if (blk < nb) {
        if (ENERGY) {
            fa[T.lufs_e + blk] = __fdiv_rn(sum, (float)my_len);
        } else {
            fa[T.lufs_z + 2 * (uint64_t)blk] = x1;
            fa[T.lufs_z + 2 * (uint64_t)blk + 1] = x2;
        }
    }
}

struct Affine {  // s -> M s + v
    float m00, m01, m10, m11, v0, v1;
};
__device__ __forceinline__ Affine compose(const Affine& second, const Affine& first) {  // second o first
    Affine r;
    r.m00 = second.m00 * first.m00 + second.m01 * first.m10;
    r.m01 = second.m00 * first.m01 + second.m01 * first.m11;
    r.m10 = second.m10 * first.m00 + second.m11 * first.m10;
    r.m11 = second.m10 * first.m01 + second.m11 * first.m11;
    r.v0 = second.m00 * first.v0 + second.m01 * first.v1 + second.v0;
    r.v1 = second.m10 * first.v0 + second.m11 * first.v1 + second.v1;
    return r;
}

__global__ void __launch_bounds__(32) lufs_scan_kernel(const TrackDev* __restrict__ tr, const SrTables* __restrict__ srtab, const int32_t* __restrict__ sr_index,
                                                       float* fa) {
    const int t = blockIdx.x;
    const TrackDev& T = tr[t];
    if (T.status != 0 || T.lufs_nb == 0) return;
    const int lane = threadIdx.x;
    const SrTables& st = srtab[sr_index[t]];
    const Biquad q{st.kw_b0, st.kw_b1, st.kw_b2, st.kw_a1, st.kw_a2};
    const uint32_t nb = T.lufs_nb, B = T.lufs_block;
    // P = A^B: lanes 0 and 1 run the homogeneous recurrence from the two basis states
    float h1 = lane == 0 ? 1.0f : 0.0f, h2 = lane == 1 ? 1.0f : 0.0f;
    if (lane < 2)
        for (uint32_t i = 0; i < B; ++i) biquad_step(q, 0.0f, h1, h2);
    Affine P;
    P.m00 = __shfl_sync(0xffffffffu, h1, 0);
    P.m10 = __shfl_sync(0xffffffffu, h2, 0);
    P.m01 = __shfl_sync(0xffffffffu, h1, 1);
    P.m11 = __shfl_sync(0xffffffffu, h2, 1);
    P.v0 = P.v1 = 0.0f;
    // every full block c maps its start state to the next one by (P, z_c); lane l owns blocks [a, b)
    const uint32_t n_maps = nb - 1;  // the last block's end state is never needed
    const uint32_t per = (n_maps + 31) / 32;
    const uint32_t a = min(lane * per, n_maps), b = min(a + per, n_maps);
    const float* z = fa + T.lufs_z;
    Affine loc{1.0f, 0.0f, 0.0f, 1.0f, 0.0f, 0.0f};
    for (uint32_t c = a; c < b; ++c) {
        Affine m = P;
        m.v0 = z[2 * (uint64_t)c];
        m.v1 = z[2 * (uint64_t)c + 1];
        loc = compose(m, loc);
    }
    // inclusive warp scan of the per-lane composites (Hillis-Steele over affine composition)
    Affine inc = loc;
    for (int o = 1; o < 32; o <<= 1) {
        Affine up;
        up.m00 = __shfl_up_sync(0xffffffffu, inc.m00, o);
        up.m01 = __shfl_up_sync(0xffffffffu, inc.m01, o);
        up.m10 = __shfl_up_sync(0xffffffffu, inc.m10, o);
        up.m11 = __shfl_up_sync(0xffffffffu, inc.m11, o);
        up.v0 = __shfl_up_sync(0xffffffffu, inc.v0, o);
        up.v1 = __shfl_up_sync(0xffffffffu, inc.v1, o);
        if (lane >= o) inc = compose(inc, up);
    }
    // state entering this lane's first block = exclusive prefix applied to the zero state
    float s0 = __shfl_up_sync(0xffffffffu, inc.v0, 1), s1 = __shfl_up_sync(0xffffffffu, inc.v1, 1);
    if (lane == 0) s0 = s1 = 0.0f;
    float* sout = fa + T.lufs_s;
    for (uint32_t c = a; c < b; ++c) {
        sout[2 * (uint64_t)c] = s0;
        sout[2 * (uint64_t)c + 1] = s1;
        const float n0 = P.m00 * s0 + P.m01 * s1 + z[2 * (uint64_t)c];
        const float n1 = P.m10 * s0 + P.m11 * s1 + z[2 * (uint64_t)c + 1];
        s0 = n0;
        s1 = n1;
    }
    // lane 31's range always ends at n_maps, so after its loop it holds the state entering the last block
    if (lane == 31) {
        sout[2 * (uint64_t)n_maps] = s0;
        sout[2 * (uint64_t)n_maps + 1] = s1;
    }
}

constexpr int SRMS_SEG = 16;  // hop-blocks per segment of the streamed frame-RMS (framed.cuh)
// Frames of FRAME samples at hop FRAME / 2 (silence.rs:144)
template <int FRAME>
__global__ void __launch_bounds__(128) silence_rms_kernel(const float* __restrict__ x, TrackDev* tr, float* fa) {
    __shared__ float tiles[4][2][16][33];
    const int t = blockIdx.y;
    const TrackDev& T = tr[t];
    const uint32_t nf = T.Fsil;
    if (T.n < FRAME) {  // one short frame (silence.rs:154-169 on a track shorter than the frame): the tile scheme with its length-aware divisor
        if (blockIdx.x == 0 && threadIdx.x < 32 && nf > 0)
            framed_rms_warp<FRAME>(x + T.off, T.n, T.gain, FRAME / 2, 0, nf, reinterpret_cast<float(*)[33]>(&tiles[0][0][0][0]), fa + T.sil_rms);
        return;
    }
    const uint32_t seg_first = (blockIdx.x * 4 + (threadIdx.x >> 5)) * 16;  // 16 segments per warp (2 lanes each)
    if (seg_first * SRMS_SEG >= nf) return;
    framed_rms_stream_warp<FRAME, FRAME / 2, SRMS_SEG>(x + T.off, T.n, T.gain, nf, seg_first, tiles[threadIdx.x >> 5], fa + T.sil_rms);
}

// detect_and_trim region logic — silence.rs:171-256.  One CTA per track.
// Only two of the reference's silence regions can move the trim points: the run that starts at frame 0 (always
// kept: `sil_start == 0`) and the run that reaches the end of the track (kept when it is long enough or starts at
// 0).  They are determined by the first and the last non-silent frame, two order-free index reductions.
__global__ void __launch_bounds__(256) trim_kernel(TrackDev* tr, const float* fa, int n_tracks, DevCfg cfg) {
    __shared__ uint32_t s_first, s_last;
    const int t = blockIdx.x;
    if (t >= n_tracks) return;
    TrackDev& T = tr[t];
    const uint64_t n = T.n;
    const uint32_t nf = T.Fsil;
    const uint32_t hop = cfg.frame / 2;
    if (threadIdx.x == 0) {
        s_first = 0xffffffffu;  // first non-silent frame
        s_last = 0u;            // last non-silent frame + 1
    }
    __syncthreads();
    if (cfg.enable_trim) {
        const float* rms = fa + T.sil_rms;
        uint32_t lf = 0xffffffffu, ll = 0u;
        for (uint32_t f = threadIdx.x; f < nf; f += blockDim.x)
            if (!(rms[f] <= cfg.silence_thr_linear)) {
                lf = min(lf, f);
                ll = max(ll, f + 1);
            }
        for (int o = 16; o > 0; o >>= 1) {
            lf = min(lf, __shfl_xor_sync(0xffffffffu, lf, o));
            ll = max(ll, __shfl_xor_sync(0xffffffffu, ll, o));
        }
        if ((threadIdx.x & 31) == 0) {
            atomicMin(&s_first, lf);
            atomicMax(&s_last, ll);
        }
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    uint64_t ts = 0, te = n;
    if (cfg.enable_trim && nf > 0) {
        const uint32_t min_samples = as_u32(__fmul_rn(__fdiv_rn((float)cfg.silence_min_ms, 1000.0f), (float)T.sr));
        const uint32_t min_frames = (min_samples + hop - 1) / hop;
        const uint32_t lead_end = s_first == 0xffffffffu ? nf : s_first;  // frames [0, lead_end) are silent
        const uint32_t trail_start = s_last;                               // frames [trail_start, nf) are silent
        if (lead_end > 0) ts = lead_end < nf ? (uint64_t)lead_end * hop : n;
        if (trail_start < nf && (nf - trail_start >= min_frames || trail_start == 0)) te = (uint64_t)trail_start * hop;
        if (ts > te) ts = te;  // trim_start.min(trim_end); trim_end.max(trim_start)
        if (!(ts < te && te <= n)) { ts = 0; te = 0; }
    }
    T.trim_start = ts;
    T.trim_end = te;
    const uint64_t m = te - ts;
    T.m = m;
    const uint32_t hops[N_HOPS] = {512, 256, 1024};
    for (int h = 0; h < N_HOPS; ++h) T.F[h] = frames_of(m, cfg.frame, hops[h]);
    T.F[SLOT_BASE_ALT] = frames_of(m, cfg.frame, cfg.hop);
    T.F[SLOT_PERC] = T.F[cfg.bs];
    T.Fk = frames_of(m, cfg.key_frame, cfg.key_hop);
    if (m == 0 && T.status == 0) {
        T.status = STRATUM_PROCESSING_ERROR;
        T.err_code = 3;  // "Audio is entirely silent after trimming" (lib.rs:143-147)
    }
}

void launch_peak(const WaveCtx& c) {
    if (c.cfg.enable_normalization) {
        uint64_t per = (c.max_n + 255) / 256;
        unsigned gx = (unsigned)((per + 63) / 64);  // ~64 float4-less iterations per thread
        if (gx < 1) gx = 1;
        if (gx > 2048) gx = 2048;
        peak_kernel<<<dim3(gx, c.n_tracks), 256, 0, c.stream>>>(c.samples, c.tracks);
        count_launch("preprocess");
        if (c.cfg.normalization == STRATUM_NORM_RMS) {
            rms_seq_kernel<<<c.n_tracks, 32, 0, c.stream>>>(c.samples, c.tracks);
            count_launch("preprocess");
        } else if (c.cfg.normalization == STRATUM_NORM_LOUDNESS && c.max_lufs_nb > 0) {
            const dim3 g((c.max_lufs_nb + 127) / 128, c.n_tracks);
            lufs_block_kernel<false><<<g, 128, 0, c.stream>>>(c.samples, c.tracks, c.srtab, c.sr_index, c.fa);
            lufs_scan_kernel<<<c.n_tracks, 32, 0, c.stream>>>(c.tracks, c.srtab, c.sr_index, c.fa);
            lufs_block_kernel<true><<<g, 128, 0, c.stream>>>(c.samples, c.tracks, c.srtab, c.sr_index, c.fa);
            count_launch("preprocess");
            count_launch("preprocess");
            count_launch("preprocess");
        }
    }
}

void launch_gain(const WaveCtx& c, const float* d_lufs_gain) {
    gain_kernel<<<(c.n_tracks + 127) / 128, 128, 0, c.stream>>>(c.tracks, c.n_tracks, c.cfg, d_lufs_gain);
    count_launch("preprocess");
}

void launch_silence_trim(const WaveCtx& c) {
    if (c.cfg.enable_trim && c.max_Fsil > 0) {
        const dim3 grid((c.max_Fsil + SRMS_SEG * 64 - 1) / (SRMS_SEG * 64), c.n_tracks);
        with_frame(c.cfg.frame, [&](auto fc) { silence_rms_kernel<decltype(fc)::F><<<grid, 128, 0, c.stream>>>(c.samples, c.tracks, c.fa); });
        count_launch("preprocess");
    }
    trim_kernel<<<c.n_tracks, 256, 0, c.stream>>>(c.tracks, c.fa, c.n_tracks, c.cfg);
    count_launch("preprocess");
}

}  // namespace sb
