// PCM sample conversion shared by the mono mixdown (k_synth.cu) and the loudness measurement (k_loudness.cu).
#pragma once
#include "common.cuh"

namespace sb {

// Sample idx of interleaved PCM in format fmt (STRATUM_PCM_*) -> f32 with the reference decoder's arithmetic
// (examples/analyze_batch.rs:70-165): u8 (s - 128) / 128; s16 s / 32768; s24 s / 8388608; s32 s as f32 / 2147483648; f32 as is;
// f64 as f32.  The integer scalings are divisions by powers of two, i.e. exact multiplications.
__device__ __forceinline__ float pcm_sample(const unsigned char* __restrict__ p, uint64_t idx, uint32_t fmt) {
    switch (fmt) {
        case STRATUM_PCM_U8: return __fmul_rn(__fsub_rn((float)p[idx], 128.0f), 0.0078125f);
        case STRATUM_PCM_S16: {
            const unsigned char* q = p + 2 * idx;
            const int16_t v = (int16_t)((uint16_t)q[0] | ((uint16_t)q[1] << 8));
            return __fmul_rn((float)v, 3.0517578125e-05f);
        }
        case STRATUM_PCM_S24: {
            const unsigned char* q = p + 3 * idx;
            int32_t v = (int32_t)((uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16));
            v = (v << 8) >> 8;  // sign-extend 24 -> 32
            return __fmul_rn((float)v, 1.1920928955078125e-07f);
        }
        case STRATUM_PCM_S32: {
            const unsigned char* q = p + 4 * idx;
            const int32_t v = (int32_t)((uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24));
            return __fmul_rn((float)v, 4.656612873077393e-10f);
        }
        case STRATUM_PCM_F32: {
            const unsigned char* q = p + 4 * idx;
            return __uint_as_float((uint32_t)q[0] | ((uint32_t)q[1] << 8) | ((uint32_t)q[2] << 16) | ((uint32_t)q[3] << 24));
        }
        default: {  // STRATUM_PCM_F64
            const unsigned char* q = p + 8 * idx;
            unsigned long long u = 0;
#pragma unroll
            for (int k = 0; k < 8; ++k) u |= (unsigned long long)q[k] << (8 * k);
            return (float)__longlong_as_double((long long)u);
        }
    }
}

}  // namespace sb
