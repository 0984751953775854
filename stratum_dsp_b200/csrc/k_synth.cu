// Device-side synthetic track generator (SURVEY §8d, tests/synth.py): click train + triad.
// Used by bench.py so that 1024 distinct 3-minute tracks (32.5 GB) never exist on the host.
// Not part of the analysis path; evaluated in double like the numpy generator, rounded once to f32.
#include "kernels.h"
#include "pcm.cuh"

namespace sb {

__global__ void __launch_bounds__(256) synth_kernel(float* __restrict__ out, uint64_t n_samples, uint32_t sr, const float* __restrict__ params5) {
    const uint32_t trk = blockIdx.y;
    const float* p = params5 + (uint64_t)trk * 5;
    const double bpm = p[0];
    const int tonic = (int)p[1], minor = (int)p[2];
    const double phase = p[3], amp = p[4];
    const double two_pi = 6.283185307179586476925286766559;
    const double f0 = 261.6255653005986 * exp2((double)tonic / 12.0);
    const double f1 = f0 * exp2((minor ? 3.0 : 4.0) / 12.0), f2 = f0 * exp2(7.0 / 12.0);
    const double period = 60.0 / bpm * (double)sr;
    const long long clen = (long long)(0.005 * (double)sr);
    float* o = out + (uint64_t)trk * n_samples;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_samples; i += (uint64_t)gridDim.x * blockDim.x) {
        const double t = (double)i / (double)sr;
        double x = amp * (sin(two_pi * f0 * t) + sin(two_pi * f1 * t) + sin(two_pi * f2 * t));
        // latest click start s_k = rint((phase + k) * period) <= i
        long long k = (long long)floor((double)i / period - phase) + 1;
        for (int tries = 0; tries < 3 && k >= 0; ++tries, --k) {
            const long long s = (long long)rint((phase + (double)k) * period);
            if (s <= (long long)i) {
                const long long d = (long long)i - s;
                if (d < clen) {
                    const double ct = (double)d / (double)sr;
                    x += 0.8 * sin(two_pi * 1000.0 * ct) * exp(-ct / 0.001);
                }
                break;
            }
        }
        o[i] = (float)x;
    }
}

// Interleaved PCM -> mono f32 with the reference decoder's arithmetic (examples/analyze_batch.rs:70-165): every channel sample is
// converted on its own (pcm_sample), the channel values are summed left to right in f32 starting from 0.0 and divided by the channel
// count.  The mean over the channels is a true division unless the count is 1.
// One grid row per track; formats and channel counts are per track (STRATUM_PCM_*).
__global__ void __launch_bounds__(256) pcm_to_mono_kernel(const unsigned char* __restrict__ pcm, float* __restrict__ out, const uint64_t* __restrict__ byte_off,
                                                          const uint64_t* __restrict__ out_off, const uint32_t* __restrict__ channels,
                                                          const uint32_t* __restrict__ formats) {
    const uint32_t trk = blockIdx.y;
    const uint32_t C = channels[trk], fmt = formats[trk];
    const uint64_t frames = out_off[trk + 1] - out_off[trk];
    const unsigned char* p = pcm + byte_off[trk];
    float* o = out + out_off[trk];
    const bool s16_aligned = fmt == STRATUM_PCM_S16 && (reinterpret_cast<uintptr_t>(p) & 1u) == 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < frames; i += (uint64_t)gridDim.x * blockDim.x) {
        if (C == 1) {
            o[i] = s16_aligned ? __fmul_rn((float)reinterpret_cast<const int16_t*>(p)[i], 3.0517578125e-05f) : pcm_sample(p, i, fmt);
        } else {
            float acc = 0.0f;
            for (uint32_t ch = 0; ch < C; ++ch) acc = __fadd_rn(acc, pcm_sample(p, i * C + ch, fmt));
            o[i] = __fdiv_rn(acc, (float)C);
        }
    }
}

void launch_pcm_to_mono(cudaStream_t s, const void* d_pcm, float* d_out, const uint64_t* d_byte_off, const uint64_t* d_out_off, const uint32_t* d_channels,
                        const uint32_t* d_formats, uint32_t n_tracks, uint64_t max_frames) {
    if (n_tracks == 0 || max_frames == 0) return;
    unsigned gx = (unsigned)((max_frames + 256 * 8 - 1) / (256 * 8));
    if (gx > 8192) gx = 8192;
    pcm_to_mono_kernel<<<dim3(gx, n_tracks), 256, 0, s>>>(static_cast<const unsigned char*>(d_pcm), d_out, d_byte_off, d_out_off, d_channels, d_formats);
    count_launch("pcm");
}

// ---- self-check of the range-restricted divisions of common.cuh against IEEE division (test instrumentation) ----------------
__device__ __forceinline__ uint32_t mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352du; x ^= x >> 15; x *= 0x846ca68bu; x ^= x >> 16;
    return x;
}
// float with a uniformly random significand and a binary exponent drawn from [elo, ehi]
__device__ __forceinline__ float rnd_float(uint32_t h, int elo, int ehi) {
    const uint32_t man = h & 0x7fffffu;
    const int e = elo + (int)((h >> 23) % (uint32_t)(ehi - elo + 1));
    return __uint_as_float(((uint32_t)(e + 127) << 23) | man);
}
__global__ void division_check_kernel(uint64_t n, uint32_t seed, unsigned long long* bad) {
    unsigned long long b0 = 0, b1 = 0, b2 = 0;
    for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t h1 = mix32((uint32_t)i ^ seed), h2 = mix32(h1 + 0x9e3779b9u + (uint32_t)(i >> 32)), h3 = mix32(h2 ^ 0x85ebca6bu);
        // div_by_25_rn: any magnitude >= 1e-30, both signs
        float a = rnd_float(h1, -99, 127);
        if (h2 & 1u) a = -a;
        if (__float_as_uint(div_by_25_rn(a)) != __float_as_uint(__fdiv_rn(a, 25.0f))) ++b0;
        // div_rn_inrange: d in [2^-40, 2^60], a in [2^-60 d, 2 d] (the mask quotient hp / (hp + rp + 1e-12) lies in [0, 1])
        const float d = rnd_float(h2, -40, 60);
        const float q = rnd_float(h3, -60, 0);
        const float num = __fmul_rn(d, q);
        if (__float_as_uint(div_rn_inrange(num, d)) != __float_as_uint(__fdiv_rn(num, d))) ++b1;
        // div_by_rcp_rn: frame-constant divisor b with y = RN(1/b), significand not all ones, a in [2^-60 b, b]
        float bb = rnd_float(h3 ^ h1, -60, 60);
        if ((__float_as_uint(bb) & 0x7fffffu) == 0x7fffffu) bb = __uint_as_float(__float_as_uint(bb) - 1u);
        const float aa = __fmul_rn(bb, rnd_float(h1 ^ 0x5bd1e995u, -60, -1));
        if (__float_as_uint(div_by_rcp_rn(aa, bb, __frcp_rn(bb))) != __float_as_uint(__fdiv_rn(aa, bb))) ++b2;
    }
    if (b0) atomicAdd(bad + 0, b0);
    if (b1) atomicAdd(bad + 1, b1);
    if (b2) atomicAdd(bad + 2, b2);
}
int check_divisions(cudaStream_t s, uint64_t n, uint32_t seed, unsigned long long* d_bad3) {
    cudaMemsetAsync(d_bad3, 0, 3 * sizeof(unsigned long long), s);
    division_check_kernel<<<148 * 8, 256, 0, s>>>(n, seed, d_bad3);
    count_launch("division_check");
    return cudaGetLastError() == cudaSuccess ? 0 : -1;
}

// FP32 FMA microbenchmark for the second roofline denominator (SURVEY §8d: the non-tensor FP32 peak is not in
// MEASURED_PEAKS.json): 8 independent FMA chains per thread, 2 flops per FMA.
__global__ void __launch_bounds__(256) fma_peak_kernel(float* out, int iters) {
    float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.0f, a2 = a0 + 2.0f, a3 = a0 + 3.0f, a4 = a0 + 4.0f, a5 = a0 + 5.0f, a6 = a0 + 6.0f, a7 = a0 + 7.0f;
    const float m = 0.999f, c = 1e-3f;
    for (int i = 0; i < iters; ++i) {
        a0 = __fmaf_rn(a0, m, c); a1 = __fmaf_rn(a1, m, c); a2 = __fmaf_rn(a2, m, c); a3 = __fmaf_rn(a3, m, c);
        a4 = __fmaf_rn(a4, m, c); a5 = __fmaf_rn(a5, m, c); a6 = __fmaf_rn(a6, m, c); a7 = __fmaf_rn(a7, m, c);
    }
    const float r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
    if (r == 123.456f) out[0] = r;  // keeps the chains alive
}

double measure_fp32_peak_tflops(cudaStream_t s, float* d_scratch) {
    const int blocks = 148 * 8, threads = 256, iters = 1 << 14;
    fma_peak_kernel<<<blocks, threads, 0, s>>>(d_scratch, 1 << 8);  // warm-up
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    cudaEventRecord(a, s);
    fma_peak_kernel<<<blocks, threads, 0, s>>>(d_scratch, iters);
    cudaEventRecord(b, s);
    cudaEventSynchronize(b);
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    if (!(ms > 0.0f)) return 0.0;
    return (double)blocks * threads * 8.0 * 2.0 * iters / (ms * 1e-3) / 1e12;
}

void launch_synth(cudaStream_t s, float* d_out, uint32_t n_tracks, uint64_t n_samples, uint32_t sr, const float* d_params5) {
    if (n_tracks == 0 || n_samples == 0) return;
    unsigned gx = (unsigned)((n_samples + 256 * 16 - 1) / (256 * 16));
    if (gx > 4096) gx = 4096;
    synth_kernel<<<dim3(gx, n_tracks), 256, 0, s>>>(d_out, n_samples, sr, d_params5);
    count_launch("synth");
}

}  // namespace sb
