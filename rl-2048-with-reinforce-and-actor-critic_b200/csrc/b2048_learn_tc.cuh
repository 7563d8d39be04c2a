// b2048_learn_tc.cuh — pieces shared by the tensor-core training kernels (b2048_learn_tc.cu: single-bf16 path and the
// dW GEMMs; b2048_learn_hp.cu: the float32-grade split-fp16 path): activation-image layouts and the dW GEMM launcher.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "b2048_internal.h"
#include "b2048_tc.cuh"

namespace b2 {

constexpr int ACT_TILE_BYTES = 32768;     // activation image of 64 samples: 4 slabs x [64 rows x 128 B]
constexpr int ACT_SLAB_BYTES = 8192;
constexpr int SMALL_TILE_BYTES = 2048;    // small K-major image of 64 samples: [16 rows x 128 B]

// byte offset of (sample row r of the chunk, slab, 16-byte chunk) inside an activation image
__device__ __forceinline__ size_t act_off(int64_t r, int slab, int chunk) {
    return (size_t)(r >> 6) * ACT_TILE_BYTES + (size_t)slab * ACT_SLAB_BYTES + (size_t)(r & 63) * 128 +
           (size_t)((chunk ^ (int)(r & 7)) << 4);
}
// byte offset of element (row j, sample r) inside a small K-major image
__device__ __forceinline__ size_t small_off(int64_t r, int j) {
    return (size_t)(r >> 6) * SMALL_TILE_BYTES + (size_t)j * 128 + (size_t)(((int)((r & 63) >> 3) ^ (j & 7)) << 4) +
           (size_t)(r & 7) * 2;
}
// slab g of the [128 rows x 4 slabs] shared-memory tile at sA2 -> the two 64-row tiles of a global activation image
__device__ __forceinline__ void store_act_slab(uint8_t* img, int64_t tile, uint32_t sA2, int g) {
#pragma unroll
    for (int half = 0; half < 2; ++half) {
        uint8_t* dst = img + (size_t)(tile * 2 + half) * ACT_TILE_BYTES + (size_t)g * ACT_SLAB_BYTES;
        bulk_store(dst, sA2 + (uint32_t)g * 16384u + (uint32_t)half * 8192u, (uint32_t)ACT_SLAB_BYTES);
    }
}

struct AtbArgs {
    const uint8_t* A;       // activation image (MN-major A operand: M = 256 features, K = samples)
    const uint8_t* B;       // NB == 256: activation image (MN-major B); NB == 16: small K-major image
    int64_t tiles64;
    float* C;               // C[m * ldm + n * ldn] += sum_s A[s][m] B[s][n]   for n < n_valid
    int ldm, ldn, n_valid;
    float* colsum;          // optional [256]: += column sums of the staged A (colsum_of_b == 0) or B image
    int colsum_of_b;
    int f16;                // operands are fp16 (split-precision path) instead of bf16
    const float* inv_scale; // optional device float: results are multiplied by it (undoes the fp16 path's loss scale)
};

template <int NB>
struct AtbCfg {
    static constexpr int kBBytes = NB == 256 ? ACT_TILE_BYTES : SMALL_TILE_BYTES;
    static constexpr int kStageBytes = ACT_TILE_BYTES + kBBytes;
    static constexpr int kStages = NB == 256 ? 3 : 4;
    static constexpr int kBar = kStages * kStageBytes;
    static constexpr int kSmem = kBar + 128;
    static constexpr uint32_t kTmemCols = NB == 256 ? 512u : 32u;
};

template <int NB>
int launch_atb(b2048_handle* h, const AtbArgs& a, cudaStream_t stream);

}  // namespace b2
