// b2048_tc.cuh — shared pieces of the tcgen05 / TMEM kernels (policy forward: b2048_policy_tc.cu; training
// forward + backward and the dW GEMMs: b2048_learn_tc.cu, b2048_learn_hp.cu; the generic MLP: b2048_mlp_gen.cu): the bf16
// weight image layout and the shared-memory / instruction descriptors.  The PTX wrappers are in b2048_ptx.cuh.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "b2048_ptx.cuh"

namespace b2 {

constexpr int TC_M = 128;          // boards per tile = TMEM lanes
constexpr int TC_H = 256;          // hidden width (both layers)
constexpr int TC_K1 = 16;          // input width
constexpr int TC_N3 = 16;          // head width padded to the UMMA minimum for M = 128

// ---- shared-memory image (byte offsets).  SW128 K-major slabs must be 1024-byte aligned.
constexpr int IMG_W2 = 0;                          // 4 slabs [256 rows x 128 B] = 131072 B (SWIZZLE_128B, K-major)
constexpr int IMG_W1 = 131072;                     // [32 row-groups][2 k-chunks][8 rows][16 B] = 8192 B (no swizzle)
constexpr int IMG_BIAS = IMG_W1 + 8192;            // same layout: k = 0 -> b1[n], k = 1 -> b2[n], rest 0
constexpr int IMG_W3 = IMG_BIAS + 8192;            // 4 slabs [16 rows x 128 B] = 8192 B (SWIZZLE_128B), rows 4..15 zero
constexpr int IMG_B3 = IMG_W3 + 8192;              // float [4]
constexpr int IMG_ONES1 = IMG_B3 + 256;            // [2 k-chunks][8 rows][16 B] = 256 B: every row = e0
constexpr int IMG_ONES2 = IMG_ONES1 + 256;         // every row = e1
constexpr int IMG_BYTES = IMG_ONES2 + 256;         // 156416
// ---- per-CTA working buffers after the image
constexpr int SM_A2 = ((IMG_BYTES + 1023) / 1024) * 1024;   // 4 slabs [128 rows x 128 B] = 65536 B (SWIZZLE_128B)
constexpr int SM_A1 = SM_A2 + 65536;                        // [16 row-groups][2][8][16 B] = 4096 B (no swizzle)
constexpr int SM_BAR = SM_A1 + 4096;                        // mbarriers + tmem base
constexpr int SM_TOTAL2 = SM_BAR + 256;
static_assert(IMG_W3 % 1024 == 0 && SM_A2 % 1024 == 0 && IMG_BYTES % 16 == 0, "operand alignment");
static_assert(SM_TOTAL2 <= 232448, "exceeds the 227 KB shared memory of an sm_100 CTA");

// ------------------------------------------------------------------------------------------------ descriptors
// SWIZZLE_128B K-major operand: rows of 128 B, 8-row groups 1024 B apart (SBO), version 1 (sm_100)
__device__ __forceinline__ uint64_t desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// no-swizzle K-major operand with K = 16: core matrix = 8 rows x 16 B (128 B contiguous);
// the second 16-byte K chunk is LBO = 128 B away, the next 8-row group SBO = 256 B away
__device__ __forceinline__ uint64_t desc_nosw_k16(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(128 >> 4) << 16) | ((uint64_t)(256 >> 4) << 32) | (1ull << 46);
}
// constant A operand (ONES1 / ONES2): chunk 1 is LBO = 128 B after chunk 0, and SBO = 0 makes every 8-row group
// read the same 128-byte core matrix
__device__ __forceinline__ uint64_t desc_ones(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(128 >> 4) << 16) | (1ull << 46);
}
constexpr uint32_t DH_SW = 0x40004040u;     // upper word of desc_sw128: SBO 1024, version 1, 128-byte swizzle
constexpr uint32_t DH_NOSW = 0x4010u;       // desc_nosw_k16: SBO 256, version 1
constexpr uint32_t DH_ONES = 0x4000u;       // desc_ones: SBO 0, version 1
__device__ __forceinline__ uint32_t dlo_sw(uint32_t saddr) { return (saddr >> 4) | (1u << 16); }
__device__ __forceinline__ uint32_t dlo_ns(uint32_t saddr) { return (saddr >> 4) | (8u << 16); }

// MN-major SWIZZLE_128B operand (the contiguous dimension is M or N, not K): a [K rows][64 MN elements = 128 B] atom
// of 8 K-rows (1024 B); the next 8 K-rows are SBO = 1024 B away, the next 64 MN elements LBO bytes away.
__device__ __forceinline__ uint64_t desc_sw128_mn(uint32_t saddr, uint32_t lbo_bytes) {
    return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo_bytes >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) |
           (1ull << 46) | (2ull << 61);
}

// kind::f16 instruction descriptors: D fp32, A and B K-major (or with the MN-major bits below), M x N
__host__ __device__ constexpr uint32_t idesc_bf16(int m, int n) {   // A/B bf16
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__host__ __device__ constexpr uint32_t idesc_f16(int m, int n) {    // A/B fp16
    return (1u << 4) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
constexpr uint32_t kIdescAMn = 1u << 15;   // instruction-descriptor bit: A is MN-major
constexpr uint32_t kIdescBMn = 1u << 16;   // instruction-descriptor bit: B is MN-major
constexpr uint32_t kIdesc = idesc_bf16(TC_M, TC_H);
constexpr uint32_t kIdescHead = idesc_bf16(TC_M, TC_N3);

}  // namespace b2
