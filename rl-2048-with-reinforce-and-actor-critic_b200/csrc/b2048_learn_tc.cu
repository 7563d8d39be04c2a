// b2048_learn_tc.cu — K6 on the 5th-generation tensor cores, SINGLE-bf16 operands (precision 1, an explicit opt-in since
// round 2), and the dW GEMM kernels shared with the default path: the policy-gradient / value-gradient accumulation of
// update_batch (src/reinforce_agent.py:403-555, _backpropagation :639-678) for the runner-default network shape
// (16 -> 256 -> 256 -> n_out <= 4, ReLU), fp32 accumulation in TMEM.  The kernels are exact against a restatement of the same
// bf16 roundings (1e-4), but a bf16 FORWARD pass flips ReLU units near zero relative to the reference's float32 arithmetic:
// 3-30 % error on cancelling gradients.  The default tensor-core path (split-fp16 forward, b2048_learn_hp.cu) meets the 1e-2
// bar; atb_tc_kernel below serves both (bf16 or fp16 images).
//
// Two kernels per chunk of samples:
//
//  fb_tc_kernel  (forward + backward deltas; one CTA = 128 samples = 128 TMEM lanes, persistent over tiles)
//      D1 = A1 W1^T + b1            -> H1 = relu(D1)        (epilogue 1: smem operand + global image + sign bits)
//      D2 = H1 W2^T + b2            -> H2 = relu(D2)        (epilogue 2: same)
//      D3 = H2 W3^T                 -> logits -> masked softmax -> d3 = coef (onehot(a) - pi)   (I/O warps)
//      D5 = d3 W3^T                 one MMA (K = 16): the head's W3 image read as an MN-major B operand
//      DL2 = D5 . [z2 > 0]                                                                          (epilogue 3)
//      D4 = DL2 W2                  the SAME shared-memory W2 image read as an MN-major B operand
//      DL1 = D4 . [z1 > 0]                                                                          (epilogue 4)
//    H1, H2, DL2, DL1 leave the SM as bf16 "activation images": per 64 samples, four 64-feature slabs of
//    [64 rows x 128 B] with the 128-byte swizzle already applied — byte-for-byte what the UMMA descriptors of the
//    second kernel expect, so that kernel stages them with plain bulk copies (no tensor map, no re-layout).
//
//  atb_tc_kernel<NB>  (dW = A^T B summed over samples, split over CTAs by sample range)
//      A is an activation image read as an MN-major operand (M = features, K = samples), B is either another
//      activation image (MN-major, NB = 256: dW2 = H1^T DL2) or a small K-major [16 x 64] image (NB = 16:
//      dW3 = H2^T d3 and dW1^T = DL1^T A1).  3-4 stage bulk-copy pipeline, accumulators stay in TMEM for the
//      whole sample range of the CTA and are added into the gradient with float atomics at the end.  Idle
//      warps add up the columns of the staged DL tiles for the bias gradients (no extra HBM pass).
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#include "b2048_device.cuh"
#include "b2048_internal.h"
#include "b2048_tc.cuh"
#include "b2048_learn_tc.cuh"

namespace b2 {

// ------------------------------------------------------------------------------------------------ layouts
constexpr int FB_D3A = SM_BAR + 256;      // head deltas of the tile in flight as a bf16 A operand [128 x 16], A1's layout
constexpr int FB_TOTAL = FB_D3A + 4096;
static_assert(FB_TOTAL <= 232448, "fb_tc_kernel exceeds the shared memory of an sm_100 CTA");

struct TcWorkspace {       // byte offsets inside the caller's workspace for a chunk padded to `np` samples
    int64_t h1, h2, dl2, dl1, a1t, d3t, total;
};
static TcWorkspace tc_workspace(int64_t chunk) {
    TcWorkspace w;
    const int64_t np = (chunk + TC_M - 1) / TC_M * TC_M;
    const int64_t act = np / 64 * ACT_TILE_BYTES, small = np / 64 * SMALL_TILE_BYTES;
    w.h1 = 0; w.h2 = act; w.dl2 = 2 * act; w.dl1 = 3 * act; w.a1t = 4 * act; w.d3t = 4 * act + small;
    w.total = 4 * act + 2 * small;
    return w;
}

struct FbArgs {
    const uint8_t* img;
    const uint64_t* board;
    const uint8_t* mask_flags;
    const uint8_t* action;
    const float* coef;
    uint8_t *h1, *h2, *dl2, *dl1, *a1t, *d3t;
    float* gb3;            // head bias gradient (atomics)
    int64_t n;
    int head_mode, n_out, obs_mode;
    float obs_scale;
    long long* debug_clock;   // optional phase timestamps of CTA 0's first epilogue thread (B2048_TC_DEBUG_CLOCK)
};

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {
    __nv_bfloat162 p = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&p);
}

// Epilogues 1 / 2: relu + bf16 pack of this warp's 16 columns in each of the four K slabs into the shared-memory
// operand of the next MMA.  The same bytes are the global activation image of the tile: the MMA warp streams each
// finished slab out with bulk async copies (store_act_slab), so the epilogue threads issue no global stores (a per-thread
// 16-byte store at a 128-byte stride costs 32 LSU wavefronts per instruction and was the kernel's bottleneck).
// Returns the 64 "z > 0" bits of the thread's columns (bit 16 s + 15 - i for column i of slab s).
__device__ __forceinline__ uint64_t fb_relu_store(uint32_t tcol0, uint8_t* a2_row, int row, int g, int lane, uint32_t bar0) {
    uint32_t mw[4];
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        uint32_t r[16];
        tmem_ld16(tcol0 + (uint32_t)(s * 64 + g * 16), r);
        uint32_t m = 0;
#pragma unroll
        for (int i = 0; i < 16; ++i) m = __funnelshift_l(0u - r[i], m, 1);   // z > 0  <=>  sign bit of -bits(z)
        mw[s] = m;
#pragma unroll
        for (int c = 0; c < 2; ++c) {
            uint4 v = make_uint4(relu_pack(r[c * 8 + 0], r[c * 8 + 1]), relu_pack(r[c * 8 + 2], r[c * 8 + 3]),
                                 relu_pack(r[c * 8 + 4], r[c * 8 + 5]), relu_pack(r[c * 8 + 6], r[c * 8 + 7]));
            const int sw = ((g * 2 + c) ^ (row & 7)) << 4;
            *reinterpret_cast<uint4*>(a2_row + s * 16384 + sw) = v;
        }
        fence_proxy_async_smem();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar0 + 8u * s);
    }
    return (uint64_t)(mw[0] | (mw[1] << 16)) | ((uint64_t)(mw[2] | (mw[3] << 16)) << 32);
}

__device__ __forceinline__ float bf_lo(uint32_t w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf_hi(uint32_t w) { return __uint_as_float(w & 0xFFFF0000u); }


constexpr int FB_THREADS = 512 + 32 + 128;

__global__ void __launch_bounds__(FB_THREADS, 1) fb_tc_kernel(const __grid_constant__ FbArgs args) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_BAR);
    const uint32_t bar_img = s_u32(&bars[0]), bar_a1 = s_u32(&bars[1]), bar_d1 = s_u32(&bars[2]), bar_d2 = s_u32(&bars[3]),
                   bar_d3 = s_u32(&bars[4]), bar_dl3 = s_u32(&bars[5]), bar_d4 = s_u32(&bars[6]), bar_free = s_u32(&bars[7]);
    const uint32_t bar_slab0 = s_u32(&bars[8]);     // [8..11]  H1 slab written
    const uint32_t bar_hslab0 = s_u32(&bars[12]);   // [12..15] H2 slab written
    const uint32_t bar_bslab0 = s_u32(&bars[16]);   // [16..19] DL2 slab written
    const uint32_t bar_dslab0 = s_u32(&bars[20]);   // [20..23] DL1 slab written (D4 drained for that slab)
    const uint32_t bar_d5 = s_u32(&bars[24]);       // D5 = d3 W3^T complete
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM_BAR + 208);

    if (tid == 0) {
        mbar_init(bar_img, 1);
        mbar_init(bar_a1, 4);
        mbar_init(bar_d1, 1);
        mbar_init(bar_d2, 1);
        mbar_init(bar_d3, 1);
        mbar_init(bar_dl3, 4);
        mbar_init(bar_d4, 1);
        mbar_init(bar_d5, 1);
        mbar_init(bar_free, 1);                      // A2 buffer free: the DL1 image of the tile has been streamed out
        for (int g = 0; g < 4; ++g) {
            mbar_init(bar_slab0 + 8u * g, 16);
            mbar_init(bar_hslab0 + 8u * g, 16);
            mbar_init(bar_bslab0 + 8u * g, 16);
            mbar_init(bar_dslab0 + 8u * g, 16);
        }
        mbar_init_fence();
    }
    // D1 = columns 0..255 (D3 re-uses 0..15 once D1 is drained), D2 / D4 = columns 256..511
    const uint32_t tmem_base = tmem_setup(warp == 16, tmem_slot, 512u);
    const int64_t n_tiles = (args.n + TC_M - 1) / TC_M;
    const int64_t first = blockIdx.x;

    if (warp == 16) {
        // ============================ MMA / copy warp ============================
        const uint32_t sA1 = s_u32(smem + SM_A1), sA2 = s_u32(smem + SM_A2);
        const uint32_t sW1 = s_u32(smem + IMG_W1), sW2 = s_u32(smem + IMG_W2), sW3 = s_u32(smem + IMG_W3);
        const uint64_t dBias = desc_nosw_k16(s_u32(smem + IMG_BIAS));
        const uint64_t dOnes1 = desc_ones(s_u32(smem + IMG_ONES1)), dOnes2 = desc_ones(s_u32(smem + IMG_ONES2));
        constexpr uint32_t kIdescBwd = idesc_bf16(TC_M, TC_H) | kIdescBMn;
        if (lane == 0) {
            mbar_expect_tx(bar_img, (uint32_t)IMG_BYTES);
            bulk_load_chunked<16384u>(s_u32(smem), args.img, (uint32_t)IMG_BYTES, bar_img);
            mbar_wait(bar_img, 0);
        }
        __syncwarp();
        auto issue_layer1 = [&](uint32_t ph) {
            mbar_wait(bar_a1, ph);
            tc_fence_after();
            umma_f16(tmem_base, desc_nosw_k16(sA1), desc_nosw_k16(sW1), kIdesc, 0u);
            umma_f16(tmem_base, dOnes1, dBias, kIdesc, 1u);
            umma_commit(bar_d1);
        };
        uint32_t ph = 0;
        if (lane == 0 && first < n_tiles) issue_layer1(0u);
        for (int64_t tile = first; tile < n_tiles; tile += gridDim.x) {
            if (lane == 0) {
                // ---- layer 2 (D2 = columns 256..511; the previous tile's D4 lives there until epilogue 4 is done)
                //      (its D4 was drained before the DL1 slab arrivals this warp waited for at the end of that tile)
                for (int g = 0; g < 4; ++g) {
                    mbar_wait(bar_slab0 + 8u * g, ph);
                    tc_fence_after();
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        umma_f16(tmem_base + 256u, desc_sw128(sA2 + (uint32_t)g * 16384u + (uint32_t)q * 32u),
                                 desc_sw128(sW2 + (uint32_t)g * 32768u + (uint32_t)q * 32u), kIdesc, (g | q) ? 1u : 0u);
                    store_act_slab(args.h1, tile, sA2, g);
                }
                umma_f16(tmem_base + 256u, dOnes2, dBias, kIdesc, 1u);
                bulk_commit();
                bulk_wait_read();                        // epilogue 2 overwrites H1 once bar_d2 completes
                umma_commit(bar_d2);
                // ---- head: D3 = columns 0..15 (D1 has been drained by every warp before the H1 slab arrivals)
                for (int g = 0; g < 4; ++g) {
                    mbar_wait(bar_hslab0 + 8u * g, ph);
                    tc_fence_after();
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        umma_f16(tmem_base, desc_sw128(sA2 + (uint32_t)g * 16384u + (uint32_t)q * 32u),
                                 desc_sw128(sW3 + (uint32_t)g * 2048u + (uint32_t)q * 32u), kIdescHead, (g | q) ? 1u : 0u);
                    store_act_slab(args.h2, tile, sA2, g);
                }
                bulk_commit();
                bulk_wait_read();                        // epilogue 3 overwrites H2 once bar_d3 completes
                umma_commit(bar_d3);
                // ---- backward through the head: D5 = d3 . W3^T into columns 0..255 (D1 / D3 are dead: the I/O warps have
                //      read D3).  A = d3 as bf16 [128 x 16] (K-major, A1's layout); B = the head's W3 image [j][f]
                //      read MN-major (N = f contiguous: 64-wide slabs 2048 B apart, 8 K rows = 1024 B).
                mbar_wait(bar_dl3, ph);
                tc_fence_after();
                umma_f16(tmem_base, desc_nosw_k16(s_u32(smem + FB_D3A)), desc_sw128_mn(sW3, 2048u), kIdescBwd, 0u);
                umma_commit(bar_d5);
                // ---- backward through layer 2: D4 = DL2 . W2 over K = out features; B = the W2 image [out][in]
                //      read MN-major (N = in contiguous: 64-wide slabs 32768 B apart, 8 K rows = 1024 B)
                for (int g = 0; g < 4; ++g) {
                    mbar_wait(bar_bslab0 + 8u * g, ph);
                    tc_fence_after();
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        umma_f16(tmem_base + 256u, desc_sw128(sA2 + (uint32_t)g * 16384u + (uint32_t)q * 32u),
                                 desc_sw128_mn(sW2 + (uint32_t)(g * 64 + q * 16) * 128u, 32768u), kIdescBwd,
                                 (g | q) ? 1u : 0u);
                    store_act_slab(args.dl2, tile, sA2, g);
                }
                bulk_commit();
                bulk_wait_read();                        // epilogue 4 overwrites DL2 once bar_d4 completes
                umma_commit(bar_d4);
                // ---- the next tile's layer 1 (D5 was drained by every warp before the DL2 slab arrivals)
                if (tile + gridDim.x < n_tiles) issue_layer1(ph ^ 1u);
                // ---- DL1 leaves through the same buffer; the next tile's epilogue 1 may reuse it afterwards
                for (int g = 0; g < 4; ++g) {
                    mbar_wait(bar_dslab0 + 8u * g, ph);
                    store_act_slab(args.dl1, tile, sA2, g);
                }
                bulk_commit();
                bulk_wait_read();
                mbar_arrive(bar_free);
            }
            __syncwarp();
            ph ^= 1u;
        }
        if (lane == 0) bulk_wait();   // image writes complete before exit
        __syncwarp();
    } else if (warp < 16) {
        // ============================ epilogue warps ============================
        const int q = warp & 3, g = warp >> 2;
        const int row = q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        uint8_t* a2_row = smem + SM_A2 + row * 128;
        uint32_t ph = 0;
        for (int64_t tile = first; tile < n_tiles; tile += gridDim.x) {
            const int64_t lt = (tile - first) / gridDim.x;
            const bool dbg = args.debug_clock != nullptr && blockIdx.x == 0 && tid == 0 && lt < 6;
            long long* dc = dbg ? args.debug_clock + 10 * lt : nullptr;
            if (dbg) dc[0] = clock64();
            // ---- epilogue 1: H1 (A2 is free once the previous tile's DL1 image has been streamed out)
            mbar_wait(bar_d1, ph);
            if (tile != first) mbar_wait(bar_free, ph ^ 1u);
            if (dbg) dc[1] = clock64();
            tc_fence_after();
            const uint64_t m1 = fb_relu_store(tlane, a2_row, row, g, lane, bar_slab0);
            if (dbg) dc[2] = clock64();
            // ---- epilogue 2: H2 over H1 (layer 2 has completed)
            mbar_wait(bar_d2, ph);
            if (dbg) dc[3] = clock64();
            tc_fence_after();
            const uint64_t m2 = fb_relu_store(tlane + 256u, a2_row, row, g, lane, bar_hslab0);
            if (dbg) dc[4] = clock64();
            // ---- epilogue 3: DL2 = D5 [z2 > 0] over H2 (D5 complete => the head MMAs that read H2 have completed)
            mbar_wait(bar_d5, ph);
            if (dbg) dc[5] = clock64();
            tc_fence_after();
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                uint32_t rr[16];
                tmem_ld16(tlane + (uint32_t)(s * 64 + g * 16), rr);
                const uint32_t mb = (uint32_t)(m2 >> (16 * s)) & 0xFFFFu;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    uint32_t out[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int i0 = c * 8 + 2 * k;
                        float lo = (mb >> (15 - i0)) & 1u ? __uint_as_float(rr[i0]) : 0.0f;
                        float hi = (mb >> (14 - i0)) & 1u ? __uint_as_float(rr[i0 + 1]) : 0.0f;
                        out[k] = pack_bf16(lo, hi);
                    }
                    const int sw = ((g * 2 + c) ^ (row & 7)) << 4;
                    *reinterpret_cast<uint4*>(a2_row + s * 16384 + sw) = make_uint4(out[0], out[1], out[2], out[3]);
                }
                fence_proxy_async_smem();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_bslab0 + 8u * s);
            }
            if (dbg) dc[6] = clock64();
            // ---- epilogue 4: DL1 = D4 [z1 > 0] over DL2 (the backward MMAs have completed), streamed out by the MMA warp
            mbar_wait(bar_d4, ph);
            if (dbg) dc[7] = clock64();
            tc_fence_after();
#pragma unroll
            for (int s = 0; s < 4; ++s) {
                uint32_t rr[16];
                tmem_ld16(tlane + 256u + (uint32_t)(s * 64 + g * 16), rr);
                const uint32_t mb = (uint32_t)(m1 >> (16 * s)) & 0xFFFFu;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    uint32_t out[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const int i0 = c * 8 + 2 * k;
                        float lo = (mb >> (15 - i0)) & 1u ? __uint_as_float(rr[i0]) : 0.0f;
                        float hi = (mb >> (14 - i0)) & 1u ? __uint_as_float(rr[i0 + 1]) : 0.0f;
                        out[k] = pack_bf16(lo, hi);
                    }
                    const int sw = ((g * 2 + c) ^ (row & 7)) << 4;
                    *reinterpret_cast<uint4*>(a2_row + s * 16384 + sw) = make_uint4(out[0], out[1], out[2], out[3]);
                }
                fence_proxy_async_smem();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_dslab0 + 8u * s);
            }
            if (dbg) dc[8] = clock64();
            ph ^= 1u;
        }
    } else {
        // ============================ I/O warps (17..20), one thread per sample ============================
        const int q = warp & 3;
        const int row = q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        const float* sB3 = reinterpret_cast<const float*>(smem + IMG_B3);
        uint8_t* d3a = smem + FB_D3A + (row >> 3) * 256 + (row & 7) * 16;   // this row's two 16-byte K chunks
        *reinterpret_cast<uint4*>(d3a + 128) = make_uint4(0u, 0u, 0u, 0u);    // k = 8..15 stay zero
        uint32_t ph = 0;

        auto encode_a1 = [&](int64_t tile) {
            const int64_t s = tile * TC_M + row;
            uint64_t bd = (s < args.n) ? args.board[s] : 0ull;
            uint32_t packed[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                uint32_t e0 = (uint32_t)(bd >> (8 * j)) & 0xFu, e1 = (uint32_t)(bd >> (8 * j + 4)) & 0xFu;
                float v0, v1;
                if (args.obs_mode == B2048_OBS_RAW) { v0 = e0 ? (float)(1u << e0) : 0.0f; v1 = e1 ? (float)(1u << e1) : 0.0f; }
                else { v0 = (float)e0 * args.obs_scale; v1 = (float)e1 * args.obs_scale; }
                packed[j] = pack_bf16(v0, v1);
                // transposed copy for dW1^T = DL1^T A1 (B operand [feature][sample], K-major)
                *reinterpret_cast<uint16_t*>(args.a1t + small_off(s, 2 * j)) = (uint16_t)(packed[j] & 0xFFFFu);
                *reinterpret_cast<uint16_t*>(args.a1t + small_off(s, 2 * j + 1)) = (uint16_t)(packed[j] >> 16);
            }
            uint8_t* a1 = smem + SM_A1 + (row >> 3) * 256 + (row & 7) * 16;
            *reinterpret_cast<uint4*>(a1) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
            *reinterpret_cast<uint4*>(a1 + 128) = make_uint4(packed[4], packed[5], packed[6], packed[7]);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_a1);
        };

        if (first < n_tiles) encode_a1(first);
        mbar_wait(bar_img, 0);
        for (int64_t tile = first; tile < n_tiles; tile += gridDim.x) {
            const int64_t s = tile * TC_M + row;
            const bool valid = s < args.n;
            const bool use_mask = args.mask_flags != nullptr;
            uint32_t fl = 0xFu, act = 0;
            float cf = 0.0f;
            if (valid) {
                if (use_mask) fl = args.mask_flags[s];
                if (args.action) act = args.action[s];
                cf = args.coef[s];
            }
            mbar_wait(bar_d1, ph);                                               // A1 is free
            const int64_t next = tile + gridDim.x;
            if (next < n_tiles) encode_a1(next);
            mbar_wait(bar_d3, ph);
            tc_fence_after();
            uint32_t r4[4];
            tmem_ld4(tlane, r4);
            tc_fence_before();
            float d0, d1 = 0.0f, d2 = 0.0f, d3 = 0.0f;
            if (args.head_mode == 0) {
                const float lg0 = __uint_as_float(r4[0]) + sB3[0], lg1 = __uint_as_float(r4[1]) + sB3[1];
                const float lg2 = __uint_as_float(r4[2]) + sB3[2], lg3 = __uint_as_float(r4[3]) + sB3[3];
                float m0 = (use_mask && !(fl & 1u)) ? -1e9f : lg0, m1 = (use_mask && !(fl & 2u)) ? -1e9f : lg1;
                float m2 = (use_mask && !(fl & 4u)) ? -1e9f : lg2, m3 = (use_mask && !(fl & 8u)) ? -1e9f : lg3;
                float mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));   // fast-math softmax: this thread is on the tile's critical path
                float e0 = __expf(m0 - mx), e1 = __expf(m1 - mx), e2 = __expf(m2 - mx), e3 = __expf(m3 - mx);
                float inv = __fdividef(1.0f, e0 + e1 + e2 + e3);
                d0 = cf * ((act == 0u ? 1.0f : 0.0f) - e0 * inv);                // reinforce_agent.py:340-344
                d1 = cf * ((act == 1u ? 1.0f : 0.0f) - e1 * inv);
                d2 = cf * ((act == 2u ? 1.0f : 0.0f) - e2 * inv);
                d3 = cf * ((act == 3u ? 1.0f : 0.0f) - e3 * inv);
            } else {
                d0 = cf;                                                          // value head: dLoss/dV * weight
            }
            // d3 as the bf16 A operand of D5 = d3 W3^T (k = 0..3 real), then release the MMA warp
            const uint32_t p01 = pack_bf16(d0, d1), p23 = pack_bf16(d2, d3);
            *reinterpret_cast<uint4*>(d3a) = make_uint4(p01, p23, 0u, 0u);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_dl3);
            // off the critical path: transposed bf16 copy for dW3 = H2^T d3 (rows >= n_out of the small image stay
            // zero) and the head bias gradient (sum over the warp's 32 samples)
            const uint32_t pk[2] = {p01, p23};
            const float dv[4] = {d0, d1, d2, d3};
#pragma unroll
            for (int j = 0; j < 4; ++j)
                if (j < args.n_out)
                    *reinterpret_cast<uint16_t*>(args.d3t + small_off(s, j)) = (uint16_t)(pk[j >> 1] >> (16 * (j & 1)));
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float v = dv[j];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
                if (lane == 0 && j < args.n_out && v != 0.0f) atomicAdd(args.gb3 + j, v);
            }
            ph ^= 1u;
        }
    }

    tmem_teardown(warp == 16, tmem_base, 512u);
}

// ------------------------------------------------------------------------------------------------ dW GEMM
constexpr int ATB_THREADS = 192;   // warp 0 copies, warp 1 issues the MMAs, warps 2..5 column sums + final read-out

template <int NB>
__global__ void __launch_bounds__(ATB_THREADS, 1) atb_tc_kernel(const __grid_constant__ AtbArgs args) {
    using Cfg = AtbCfg<NB>;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kBar);
    const uint32_t bar_full0 = s_u32(&bars[0]), bar_empty0 = s_u32(&bars[4]), bar_done = s_u32(&bars[8]);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + Cfg::kBar + 96);
    const bool want_colsum = args.colsum != nullptr;
    const float out_scale = args.inv_scale ? *args.inv_scale : 1.0f;

    if (tid == 0) {
        for (int i = 0; i < Cfg::kStages; ++i) {
            mbar_init(bar_full0 + 8u * i, 1);
            mbar_init(bar_empty0 + 8u * i, want_colsum ? 5 : 1);
        }
        mbar_init(bar_done, 1);
        mbar_init_fence();
    }
    const uint32_t tmem_base = tmem_setup(warp == 1, tmem_slot, Cfg::kTmemCols);
    // balanced contiguous ranges of 64-sample tiles (gridDim.x <= tiles64, so every CTA owns at least one)
    const int64_t t0 = args.tiles64 * blockIdx.x / gridDim.x, t1 = args.tiles64 * (blockIdx.x + 1) / gridDim.x;
    const int n_it = (int)(t1 - t0);

    if (warp == 0) {
        if (lane == 0) {
            for (int it = 0; it < n_it; ++it) {
                const int st = it % Cfg::kStages, use = it / Cfg::kStages;
                if (use > 0) mbar_wait(bar_empty0 + 8u * st, (uint32_t)(use - 1) & 1u);
                const uint32_t bar = bar_full0 + 8u * st;
                mbar_expect_tx(bar, (uint32_t)Cfg::kStageBytes);
                const uint8_t* ga = args.A + (size_t)(t0 + it) * ACT_TILE_BYTES;
                const uint8_t* gb = args.B + (size_t)(t0 + it) * Cfg::kBBytes;
                uint8_t* sa = smem + st * Cfg::kStageBytes;
                bulk_load_chunked<16384u>(s_u32(sa), ga, (uint32_t)ACT_TILE_BYTES, bar);
                bulk_load_chunked<16384u>(s_u32(sa + ACT_TILE_BYTES), gb, (uint32_t)Cfg::kBBytes, bar);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            // kind::f16 operand format bits (7-9: A, 10-12: B): 1 = bf16, 0 = fp16
            const uint32_t idesc = (args.f16 ? idesc_f16(128, NB) : idesc_bf16(128, NB)) | kIdescAMn | (NB == 256 ? kIdescBMn : 0u);
            for (int it = 0; it < n_it; ++it) {
                const int st = it % Cfg::kStages, use = it / Cfg::kStages;
                mbar_wait(bar_full0 + 8u * st, (uint32_t)use & 1u);
                tc_fence_after();
                const uint32_t sa = s_u32(smem + st * Cfg::kStageBytes), sb = sa + ACT_TILE_BYTES;
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {                                   // 16 samples per MMA
                    const uint64_t db = NB == 256 ? desc_sw128_mn(sb + (uint32_t)kk * 2048u, ACT_SLAB_BYTES)
                                                  : desc_sw128(sb + (uint32_t)kk * 32u);
#pragma unroll
                    for (int half = 0; half < 2; ++half)                          // features 128 half .. +127
                        umma_f16(tmem_base + (uint32_t)(half * NB),
                                 desc_sw128_mn(sa + (uint32_t)half * 16384u + (uint32_t)kk * 2048u, ACT_SLAB_BYTES), db,
                                 idesc, (it | kk) ? 1u : 0u);
                }
                umma_commit(bar_empty0 + 8u * st);
            }
            umma_commit(bar_done);
        }
        __syncwarp();
    } else {
        const int cw = warp - 2;                                                  // slab handled in the column sums
        if (want_colsum) {
            const int chunk = lane & 7, rsub = lane >> 3;
            float acc[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[e] = 0.0f;
            for (int it = 0; it < n_it; ++it) {
                const int st = it % Cfg::kStages, use = it / Cfg::kStages;
                mbar_wait(bar_full0 + 8u * st, (uint32_t)use & 1u);
                const uint8_t* x = smem + st * Cfg::kStageBytes + (args.colsum_of_b ? ACT_TILE_BYTES : 0) + cw * ACT_SLAB_BYTES;
#pragma unroll 4
                for (int r = rsub; r < 64; r += 4) {
                    const uint4 v = *reinterpret_cast<const uint4*>(x + r * 128 + ((chunk ^ (r & 7)) << 4));
                    if (args.f16) {
                        const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&v.x)), f1 = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
                        const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&v.z)), f3 = __half22float2(*reinterpret_cast<const __half2*>(&v.w));
                        acc[0] += f0.x; acc[1] += f0.y; acc[2] += f1.x; acc[3] += f1.y; acc[4] += f2.x; acc[5] += f2.y; acc[6] += f3.x; acc[7] += f3.y;
                    } else {
                        acc[0] += bf_lo(v.x); acc[1] += bf_hi(v.x); acc[2] += bf_lo(v.y); acc[3] += bf_hi(v.y);
                        acc[4] += bf_lo(v.z); acc[5] += bf_hi(v.z); acc[6] += bf_lo(v.w); acc[7] += bf_hi(v.w);
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_empty0 + 8u * st);
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                acc[e] += __shfl_xor_sync(0xFFFFFFFFu, acc[e], 8);
                acc[e] += __shfl_xor_sync(0xFFFFFFFFu, acc[e], 16);
            }
            if (lane < 8 && n_it > 0) {
#pragma unroll
                for (int e = 0; e < 8; ++e)
                    if (acc[e] != 0.0f) atomicAdd(args.colsum + cw * 64 + chunk * 8 + e, acc[e] * out_scale);
            }
        }
        // ---- read-out: TMEM lane quarter = warp % 4
        if (n_it > 0) {
            mbar_wait(bar_done, 0);
            tc_fence_after();
            const int q = warp & 3;
            const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll
            for (int half = 0; half < 2; ++half) {
                const int m = half * 128 + q * 32 + lane;
                for (int c0 = 0; c0 < NB; c0 += 16) {
                    uint32_t r[16];
                    tmem_ld16(tlane + (uint32_t)(half * NB + c0), r);
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const int n = c0 + i;
                        const float v = __uint_as_float(r[i]) * out_scale;
                        if (n < args.n_valid && v != 0.0f) atomicAdd(args.C + (size_t)m * args.ldm + (size_t)n * args.ldn, v);
                    }
                }
            }
        }
    }

    tmem_teardown(warp == 1, tmem_base, Cfg::kTmemCols);
}

template <int NB>
int launch_atb(b2048_handle* h, const AtbArgs& a, cudaStream_t stream) {
    constexpr unsigned kBit = NB == 256 ? ATTR_ATB_256 : ATTR_ATB_16;
    if (!(h->attrs & kBit)) {
        cudaError_t e = cudaFuncSetAttribute(atb_tc_kernel<NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, AtbCfg<NB>::kSmem);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(atb_tc_kernel)");
        h->attrs |= kBit;
    }
    int grid = (int)(a.tiles64 < h->num_sms ? a.tiles64 : h->num_sms);
    atb_tc_kernel<NB><<<grid, ATB_THREADS, AtbCfg<NB>::kSmem, stream>>>(a);
    return check_cuda(cudaGetLastError(), "atb_tc_kernel launch");
}

template int launch_atb<256>(b2048_handle*, const AtbArgs&, cudaStream_t);
template int launch_atb<16>(b2048_handle*, const AtbArgs&, cudaStream_t);

bool backward_tc_supported(const b2048_handle* h, const b2048_mlp_desc* mlp) {
    return fixed_tc_net(mlp) && h->smem_optin >= FB_TOTAL && h->smem_optin >= AtbCfg<256>::kSmem;
}

int64_t backward_tc_workspace_bytes(int64_t chunk) { return tc_workspace(chunk).total + 1024; }

// Same contract as the fp32 body of b2048_mlp_backward (grads accumulated, flat layout W_0, b_0, W_1, b_1, ...).
int launch_backward_tc(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags, const uint8_t* action,
                       const float* coef, const b2048_mlp_desc* mlp, float* grads, int64_t n, int head_mode,
                       uint8_t* workspace, int64_t chunk, cudaStream_t stream) {
    { int st = ensure_tc_image(h); if (st != B2048_OK) return st; }
    if (!(h->attrs & ATTR_FB_TC)) {
        cudaError_t e = cudaFuncSetAttribute(fb_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FB_TOTAL);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(fb_tc_kernel)");
        h->attrs |= ATTR_FB_TC;
    }
    launch_tc_prepare(mlp, h->tc_image, stream);
    const int n_out = mlp->dims[3];
    float *gW[B2048_MAX_LAYERS], *gb[B2048_MAX_LAYERS];
    carve_grads(mlp, grads, gW, gb);
    uint8_t* ws = reinterpret_cast<uint8_t*>(((uintptr_t)workspace + 1023) & ~(uintptr_t)1023);
    const TcWorkspace w = tc_workspace(chunk);
    long long* dbg = debug_clock_begin(h, B2048_DBG_TC_CLOCKS, stream);     // clocks of the first chunk's fb_tc_kernel
    for (int64_t c0 = 0; c0 < n; c0 += chunk) {
        const int64_t cn = (n - c0) < chunk ? (n - c0) : chunk;
        const int64_t tiles = (cn + TC_M - 1) / TC_M;
        FbArgs a;
        a.img = h->tc_image;
        a.board = board + c0;
        a.mask_flags = mask_flags ? mask_flags + c0 : nullptr;
        a.action = action ? action + c0 : nullptr;
        a.coef = coef + c0;
        a.h1 = ws + w.h1; a.h2 = ws + w.h2; a.dl2 = ws + w.dl2; a.dl1 = ws + w.dl1; a.a1t = ws + w.a1t; a.d3t = ws + w.d3t;
        a.gb3 = gb[2];
        a.n = cn;
        a.head_mode = head_mode; a.n_out = n_out; a.obs_mode = mlp->obs_mode; a.obs_scale = mlp->obs_log2_scale;
        cudaError_t e = cudaMemsetAsync(a.d3t, 0, (size_t)tiles * 2 * SMALL_TILE_BYTES, stream);
        if (e != cudaSuccess) return check_cuda(e, "cudaMemsetAsync(d3t)");
        int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
        a.debug_clock = dbg;
        fb_tc_kernel<<<grid, FB_THREADS, FB_TOTAL, stream>>>(a);
        int st = check_cuda(cudaGetLastError(), "fb_tc_kernel launch");
        if (st != B2048_OK) return st;
        if (dbg && c0 == 0) {
            long long hb[80];
            if ((st = debug_clock_read(h, hb, 80, stream)) != B2048_OK) return st;
            for (int k = 0; k < 5; ++k) {
                long long* d = hb + 10 * k;
                fprintf(stderr, "[fb clock] tile %d: wait_d1 %lld epi1 %lld wait_d2 %lld epi2 %lld wait_d3 %lld epi3 %lld wait_d4 %lld epi4 %lld | to next %lld\n",
                        k, d[1] - d[0], d[2] - d[1], d[3] - d[2], d[4] - d[3], d[5] - d[4], d[6] - d[5], d[7] - d[6], d[8] - d[7],
                        d[10] - d[0]);
            }
        }
        AtbArgs g;
        g.tiles64 = tiles * 2; g.f16 = 0; g.inv_scale = nullptr;
        // dW2 = H1^T DL2, db2 = column sums of DL2
        g.A = a.h1; g.B = a.dl2; g.C = gW[1]; g.ldm = TC_H; g.ldn = 1; g.n_valid = TC_H; g.colsum = gb[1]; g.colsum_of_b = 1;
        if ((st = launch_atb<256>(h, g, stream)) != B2048_OK) return st;
        // dW3 = H2^T d3
        g.A = a.h2; g.B = a.d3t; g.C = gW[2]; g.ldm = n_out; g.ldn = 1; g.n_valid = n_out; g.colsum = nullptr; g.colsum_of_b = 0;
        if ((st = launch_atb<16>(h, g, stream)) != B2048_OK) return st;
        // dW1^T = DL1^T A1, db1 = column sums of DL1
        g.A = a.dl1; g.B = a.a1t; g.C = gW[0]; g.ldm = 1; g.ldn = TC_H; g.n_valid = 16; g.colsum = gb[0]; g.colsum_of_b = 0;
        if ((st = launch_atb<16>(h, g, stream)) != B2048_OK) return st;
    }
    return B2048_OK;
}

}  // namespace b2

// Debug / test access to the tensor-core workspace layout: byte offsets (after 1024-byte alignment of the
// workspace pointer) of the H1, H2, DL2, DL1 activation images and the A1^T / d3^T small images, then the total.
extern "C" int b2048_backward_tc_layout(int64_t chunk, int64_t* out7) {
    B2_REQUIRE(out7 != nullptr && chunk > 0, "b2048_backward_tc_layout: bad arguments");
    const b2::TcWorkspace w = b2::tc_workspace(chunk);
    out7[0] = w.h1; out7[1] = w.h2; out7[2] = w.dl2; out7[3] = w.dl1; out7[4] = w.a1t; out7[5] = w.d3t; out7[6] = w.total;
    return B2048_OK;
}
