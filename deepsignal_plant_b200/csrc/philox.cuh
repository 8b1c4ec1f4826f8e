// N(0,1) initial states (models.py:169-176 draws torch.randn): Philox4x32-10, one subsequence per group of four
// outputs, Box-Muller via curand_normal4.  Shared by the inference path (kernels_f32.cu) and the training path
// (kernels_train.cu), so both draw the same numbers from the same seed.
#pragma once
#include <curand_kernel.h>
#include <stdint.h>

namespace dsp {

// outputs 4q .. 4q+3 of the stream (seed, stream_id), clipped at count
__device__ __forceinline__ void philox_normal_quad(float* __restrict__ out, int64_t count, uint64_t seed,
                                                   uint64_t stream_id, int64_t q) {
    int64_t base = q * 4;
    if (base >= count) return;
    curandStatePhilox4_32_10_t st;
    curand_init(seed, (unsigned long long)q, stream_id * 4ull, &st);
    float4 v = curand_normal4(&st);
    if (base + 3 < count) {
        *reinterpret_cast<float4*>(out + base) = v;
    } else {
        float tmp[4] = {v.x, v.y, v.z, v.w};
        for (int i = 0; base + i < count; ++i) out[base + i] = tmp[i];
    }
}

}  // namespace dsp
