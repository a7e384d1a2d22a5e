// rdv_policy.cuh -- small pieces shared by the actor kernels (the SB3 MlpPolicy actor 17 -> 64 -> 64 -> 6, tanh;
// main.py:39-48): the Gaussian head's Philox / Box-Muller noise.  The tensor-core forward itself (tcgen05 / TMEM,
// stand-alone and inside the rollout kernel) lives in rdv_policy_tc.cuh, the plain fp32-FMA numerics reference in
// rdv_b200.cu (policy_kernel).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "rdv_b200.h"
#include "rdv_math.cuh"

namespace rdv {

constexpr int PI_H = 64;             // hidden width (SB3 default net_arch [64, 64])

// Six N(0,1) float32 draws for (noise seed; env id, step index): Philox blocks 0x20000000 | {0,1,2}, one
// Box-Muller pair per block (the Gaussian head of SB3's DiagGaussianDistribution.sample()).
__device__ __forceinline__ void philox_normals(uint64_t seed, int64_t env_id, int64_t step_index, float (&z)[6])
{
#pragma unroll
    for (uint32_t blk = 0; blk < 3; ++blk) {
        uint32_t c[4] = {(uint32_t)env_id, (uint32_t)((uint64_t)env_id >> 32), (uint32_t)step_index,
                         0x20000000u | blk | (((uint32_t)((uint64_t)step_index >> 32) & 0x00FFFFFFu) << 4)};
        philox4x32_10(c, (uint32_t)seed, (uint32_t)(seed >> 32));
        const float u1 = ((float)(c[0] >> 8) + 0.5f) * (1.0f / 16777216.0f);      // (0, 1)
        const float u2 = ((float)(c[1] >> 8) + 0.5f) * (1.0f / 16777216.0f);
        const float r = sqrtf(-2.0f * logf(u1));
        float sn, cs;
        sincospif(2.0f * u2, &sn, &cs);
        z[2 * blk] = r * cs;
        z[2 * blk + 1] = r * sn;
    }
}

}  // namespace rdv
