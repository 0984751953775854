// Framed RMS with strict left-to-right f32 accumulation, and small block-level helpers.
#pragma once
#include "common.cuh"

namespace sb {

// ---- framed RMS with the reference's strict left-to-right f32 sum -----------------------------
// One lane per frame; a warp transposes 32x32 sample tiles through shared memory so that global
// loads stay coalesced while every lane adds its own frame's squares in sample order
// (silence.rs:159, onset/energy_flux.rs:127).
template <int FRAME>
__device__ __forceinline__ void framed_rms_warp(const float* __restrict__ x, uint64_t limit, float g, uint32_t hop, uint32_t f0, uint32_t nf,
                                                float (*tile)[33], float* out) {
    const int lane = threadIdx.x & 31;
    const uint32_t f = f0 + lane;
    float sum = 0.0f;
    for (uint32_t jb = 0; jb < FRAME; jb += 32) {
#pragma unroll 4
        for (int r = 0; r < 32; ++r) {
            uint64_t idx = (uint64_t)(f0 + r) * hop + jb + lane;
            tile[r][lane] = (f0 + r < nf && idx < limit) ? __fmul_rn(x[idx], g) : 0.0f;
        }
        __syncwarp();
#pragma unroll 8
        for (int j = 0; j < 32; ++j) {
            float v = tile[lane][j];
            sum = __fadd_rn(sum, __fmul_rn(v, v));
        }
        __syncwarp();
    }
    if (f < nf) {
        uint64_t st = (uint64_t)f * hop;
        uint64_t en = st + FRAME < limit ? st + FRAME : limit;
        // frames are always full except the single short frame of a track shorter than FRAME, where
        // the zero padding above adds exact zeros (x + 0*0 == x) and the divisor is the true length.
        float len = (float)(en - st);
        out[f] = en > st ? sqrtf(__fdiv_rn(sum, len)) : 0.0f;
    }
}


// ---- the same sums, streamed: every sample is fetched once ------------------------------------------------------
// Frames of FRAME samples at hop HOP overlap FRAME/HOP-fold; the tile scheme above fetches every sample once per frame
// that contains it (4x at hop 512), which makes the kernel L2-bandwidth bound.  Here a track is cut into segments of SEG
// hop-blocks; PH = FRAME/HOP lanes share a segment and walk its blocks together: lane p owns the frames f = p (mod PH), so at
// any block all PH lanes consume the same samples (a shared-memory broadcast), each into its own frame's running sum at a
// different position inside that frame.  A warp carries 32/PH segments; per 32 samples it issues 32/PH coalesced row loads
// (the next tile is fetched into registers while the current one is summed).  Per-frame order stays strictly left to right.
// Only full frames (tracks with at least FRAME samples); the single short frame of a shorter track stays on framed_rms_warp.
template <int FRAME, int HOP, int SEG>
__device__ __forceinline__ void framed_rms_stream_warp(const float* __restrict__ x, uint64_t limit, float g, uint32_t nf, uint32_t seg_first,
                                                       float (*tile)[32 / (FRAME / HOP)][33], float* out) {
    constexpr int PH = FRAME / HOP, GPW = 32 / PH, TILES = HOP / 32;
    static_assert(SEG % PH == 0 && HOP % 32 == 0, "segment / hop geometry");
    const int lane = threadIdx.x & 31;
    const int gq = lane / PH, p = lane % PH;
    const uint32_t tau0 = (seg_first + gq) * SEG;  // first hop-block (= first frame) of this lane's segment
    auto fetch = [&](uint32_t beta, int s, float (&r)[GPW]) {  // row q of the tile: 32 samples of block (segment q start + beta)
#pragma unroll
        for (int q = 0; q < GPW; ++q) {
            const uint64_t idx = ((uint64_t)(seg_first + q) * SEG + beta) * HOP + (uint32_t)s * 32 + lane;
            r[q] = idx < limit ? __fmul_rn(x[idx], g) : 0.0f;
        }
    };
    float nxt[GPW];
    fetch(0, 0, nxt);
    float sum = 0.0f;
    int buf = 0;
    for (uint32_t beta = 0; beta < SEG + PH - 1; ++beta) {
        // lane p joins at block p; its k-th frame spans blocks p + PH*k .. p + PH*k + PH-1 of the segment
        const int rel = (int)beta - p;
        const bool in_seg = rel >= 0 && rel < SEG;
        const uint32_t f = tau0 + p + (in_seg ? (uint32_t)(rel / PH) * PH : 0u);
        const bool active = in_seg && f < nf;
        const int c = in_seg ? rel % PH : 0;
        if (c == 0) sum = 0.0f;
        for (int s = 0; s < TILES; ++s) {
#pragma unroll
            for (int q = 0; q < GPW; ++q) tile[buf][q][lane] = nxt[q];
            __syncwarp();
            const int s2 = s + 1 < TILES ? s + 1 : 0;
            const uint32_t b2 = s + 1 < TILES ? beta : beta + 1;
            if (b2 < SEG + PH - 1) fetch(b2, s2, nxt);  // in flight while this tile is summed
            if (active) {
#pragma unroll 8
                for (int j = 0; j < 32; ++j) {
                    const float v = tile[buf][gq][j];
                    sum = __fadd_rn(sum, __fmul_rn(v, v));
                }
            }
            buf ^= 1;
        }
        if (active && c == PH - 1) out[f] = sqrtf(__fdiv_rn(sum, (float)FRAME));
    }
}

// Block-wide exclusive scan of one uint per thread (blockDim.x <= 1024, multiple of 32).
__device__ __forceinline__ uint32_t block_exclusive_scan(uint32_t v, uint32_t* total, uint32_t* warp_sums /* >= 33 */) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    uint32_t inc = v;
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t y = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += y;
    }
    if (lane == 31) warp_sums[w] = inc;
    __syncthreads();
    if (w == 0) {
        const int nw = blockDim.x >> 5;
        uint32_t s = lane < nw ? warp_sums[lane] : 0;
        uint32_t si = s;
        for (int o = 1; o < 32; o <<= 1) {
            uint32_t y = __shfl_up_sync(0xffffffffu, si, o);
            if (lane >= o) si += y;
        }
        if (lane < nw) warp_sums[lane] = si - s;
        if (lane == 31) warp_sums[32] = si;
    }
    __syncthreads();
    uint32_t res = warp_sums[w] + inc - v;
    *total = warp_sums[32];
    __syncthreads();
    return res;
}

__device__ __forceinline__ float block_max(float v, float* sm /* >= 32 */) {
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
    __syncthreads();
    const int nw = blockDim.x >> 5;
    float r = (threadIdx.x & 31) < nw ? sm[threadIdx.x & 31] : 0.0f;
    for (int o = 16; o > 0; o >>= 1) r = fmaxf(r, __shfl_xor_sync(0xffffffffu, r, o));
    __syncthreads();
    return r;
}

// top K by (value desc, index asc) of val(i) over i in [lo, hi] (values >= 0); all threads participate; result in out_idx[0..cnt).
// sval / sidx: one slot per warp.
template <int K, class F>
__device__ inline int block_topk(F val, int lo, int hi, int* out_idx, float* sval, int* sidx) {
    int cnt = 0;
    for (int r = 0; r < K; ++r) {
        float bv = -1.0f;
        int bi = 0x7fffffff;
        for (int i = lo + (int)threadIdx.x; i <= hi; i += blockDim.x) {
            bool taken = false;
            for (int q = 0; q < cnt; ++q) taken |= (out_idx[q] == i);
            if (taken) continue;
            float x = val(i);
            if (x > bv || (x == bv && i < bi)) {
                bv = x;
                bi = i;
            }
        }
        for (int o = 16; o > 0; o >>= 1) {
            float ov = __shfl_xor_sync(0xffffffffu, bv, o);
            int oi = __shfl_xor_sync(0xffffffffu, bi, o);
            if (ov > bv || (ov == bv && oi < bi)) {
                bv = ov;
                bi = oi;
            }
        }
        if ((threadIdx.x & 31) == 0) {
            sval[threadIdx.x >> 5] = bv;
            sidx[threadIdx.x >> 5] = bi;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); ++w)
                if (sval[w] > bv || (sval[w] == bv && sidx[w] < bi)) {
                    bv = sval[w];
                    bi = sidx[w];
                }
            if (bi != 0x7fffffff) out_idx[cnt] = bi;
            sidx[0] = (bi != 0x7fffffff) ? 1 : 0;
        }
        __syncthreads();
        int ok = sidx[0];
        __syncthreads();
        if (!ok) break;
        ++cnt;
    }
    return cnt;
}

template <class T>
struct SelectBits;
template <>
struct SelectBits<float> {
    using U = uint32_t;
    static __device__ __forceinline__ U bits(float x) { return __float_as_uint(x); }
    static __device__ __forceinline__ float value(U b) { return __uint_as_float(b); }
};
template <>
struct SelectBits<double> {
    using U = unsigned long long;
    static __device__ __forceinline__ U bits(double x) { return (U)__double_as_longlong(x); }
    static __device__ __forceinline__ double value(U b) { return __longlong_as_double((long long)b); }
};

// Exact k-th smallest (0-based) of n non-negative floats or doubles: MSB radix select on the bit patterns, 8 bits per
// pass (order-preserving for x >= 0).  All threads of the block call it; result broadcast.
template <class T>
__device__ inline T block_select_kth(const T* __restrict__ v, uint32_t n, uint32_t k, uint32_t* hist /* 256 */, uint32_t* bcast /* 2 */) {
    using B = SelectBits<T>;
    using U = typename B::U;
    U prefix = 0, mask = 0;
    for (int shift = 8 * (int)sizeof(U) - 8; shift >= 0; shift -= 8) {
        for (uint32_t i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
        __syncthreads();
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
            const U b = B::bits(v[i]);
            if ((b & mask) == prefix) atomicAdd(&hist[(uint32_t)(b >> shift) & 255u], 1u);
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            uint32_t acc = 0, d = 0;
            for (; d < 256; ++d) {
                if (acc + hist[d] > k) break;
                acc += hist[d];
            }
            bcast[0] = d;
            bcast[1] = k - acc;
        }
        __syncthreads();
        prefix |= (U)bcast[0] << shift;
        mask |= (U)255u << shift;
        k = bcast[1];
        __syncthreads();
    }
    return B::value(prefix);
}

}  // namespace sb
