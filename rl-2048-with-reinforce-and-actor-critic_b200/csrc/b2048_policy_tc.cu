// b2048_policy_tc.cu — K3 policy_step on the 5th-generation tensor cores (tcgen05 + TMEM), bf16 operands,
// fp32 accumulation.  Used for batches >= 4096 boards with the runner-default policy shape
// (16 -> 256 -> 256 -> 4, ReLU); everything else runs on the fp32 CUDA-core path (b2048_policy.cu).
//
// One CTA (16 epilogue warps + 1 MMA/copy warp) owns a tile of 128 boards (= the 128 TMEM lanes) and loops over tiles.
// ALL THREE layers and BOTH hidden biases run on the tensor core; the epilogues only do ReLU + bf16 pack:
//
//   A1 [128 x 16] bf16  <- packed boards (one thread per board: 16 nibbles -> 16 bf16)
//   D1 = A1 . W1^T + ONES1 . BIAS^T      2 tcgen05.mma (M128 N256 K16)          -> TMEM columns   0..255
//   A2 = bf16(relu(D1))                  tcgen05.ld 32x32b -> packed max -> st.shared, 128B-swizzled K-major slabs
//   D2 = A2 . W2^T + ONES2 . BIAS^T      16 + 1 tcgen05.mma (M128 N256 K16)     -> TMEM columns 256..511
//   H2 = bf16(relu(D2))                  same epilogue, written over A2 (free once layer 2 has completed)
//   D3 = H2 . W3^T                       16 tcgen05.mma (M128 N16 K16)          -> TMEM columns 256..271 (over D2)
//   logits = D3[:, 0:4] + b3 -> masked softmax -> inverse-CDF sample / greedy -> one action byte per board
//
// The bias trick: BIAS is a [256 x 16] operand holding b1 in k = 0 and b2 in k = 1; ONES1 / ONES2 are A operands
// whose every row is the unit vector e0 / e1.  They are 256-byte constants: their descriptors use a stride-byte-offset
// of 0 so all sixteen 8-row groups read the same core matrix.
//
// Weights arrive as a pre-arranged shared-memory IMAGE (bf16, already in the UMMA canonical layouts) that a small prep
// kernel builds from the reference-layout fp32 parameters; each CTA pulls the 153 KB image with bulk async copies
// (cp.async.bulk + mbarrier) once and keeps it resident for all of its tiles.
//
// Reference arithmetic: encode_observation / forward_logits / logits_to_probs / select_action
// (src/MLP.py:22-43, :139-196; src/reinforce_agent.py:126-192).  Parity bar for this path: 1e-2 relative.
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#include "b2048_device.cuh"
#include "b2048_internal.h"
#include "b2048_step_fast.cuh"
#include "b2048_tc.cuh"

namespace b2 {

// ------------------------------------------------------------------------------------------------ image prep
// W (reference layout [in][out] fp32) -> bf16 UMMA B operands stored [n][k] K-major.
__global__ void __launch_bounds__(256) policy_tc_prepare_kernel(const float* __restrict__ W1, const float* __restrict__ b1,
                                                                 const float* __restrict__ W2, const float* __restrict__ b2,
                                                                 const float* __restrict__ W3, const float* __restrict__ b3,
                                                                 int n_out, uint8_t* __restrict__ img) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nth = gridDim.x * blockDim.x;
    auto put = [&](size_t off, float v) { *reinterpret_cast<__nv_bfloat16*>(img + off) = __float2bfloat16_rn(v); };
    // W2: element (n, k) -> slab k/64, row n, 16-byte chunk ((k%64)/8) ^ (n%8), element k%8
    for (int idx = tid; idx < TC_H * TC_H; idx += nth) {
        int k = idx / TC_H, n = idx - k * TC_H;          // W2[k][n] is contiguous in n: coalesced reads
        int slab = k >> 6, kc = (k & 63) >> 3, ke = k & 7;
        put((size_t)IMG_W2 + (size_t)slab * 32768 + (size_t)n * 128 + (size_t)((kc ^ (n & 7)) * 16) + ke * 2, W2[idx]);
    }
    // W1 / BIAS: element (n, k), k < 16 -> row-group n/8, k-chunk k/8, row n%8, element k%8 (no swizzle)
    for (int idx = tid; idx < TC_K1 * TC_H; idx += nth) {
        int k = idx / TC_H, n = idx - k * TC_H;
        size_t off = (size_t)(n >> 3) * 256 + (size_t)(k >> 3) * 128 + (size_t)(n & 7) * 16 + (k & 7) * 2;
        put(IMG_W1 + off, W1[idx]);
        put(IMG_BIAS + off, k == 0 ? b1[n] : (k == 1 ? b2[n] : 0.0f));
    }
    // W3 (head): B operand rows j < 16 (4 real), K = 256 in four 128B-swizzled slabs of [16 rows x 128 B]
    for (int idx = tid; idx < TC_N3 * TC_H; idx += nth) {
        int j = idx / TC_H, k = idx - j * TC_H;
        int slab = k >> 6, kc = (k & 63) >> 3, ke = k & 7;
        put((size_t)IMG_W3 + (size_t)slab * 2048 + (size_t)j * 128 + (size_t)((kc ^ (j & 7)) * 16) + ke * 2,
            j < n_out ? W3[k * n_out + j] : 0.0f);
    }
    if (tid < 4) reinterpret_cast<float*>(img + IMG_B3)[tid] = tid < n_out ? b3[tid] : 0.0f;
    // ONES1 / ONES2: [k-chunk][row][8 bf16]; chunk 0 of every row holds the unit vector
    for (int idx = tid; idx < 2 * 8 * 8; idx += nth) {
        int e = idx & 7, chunk = idx >> 6;
        put(IMG_ONES1 + idx * 2, (chunk == 0 && e == 0) ? 1.0f : 0.0f);
        put(IMG_ONES2 + idx * 2, (chunk == 0 && e == 1) ? 1.0f : 0.0f);
    }
}

struct PolicyTcArgs {
    const uint8_t* img;
    const uint64_t* board;
    const uint8_t* mask_flags;
    uint8_t* action;
    float* probs;
    float* logits;
    float* head_out;          // optional [n][n_out]: raw head outputs (b2048_mlp_forward on tensor cores)
    int n_out;
    int64_t n;
    PhiloxKeys keys;
    uint64_t gid0;
    uint32_t t;
    int greedy;
    int obs_mode;
    float obs_scale;
    long long* debug_clock;   // optional: per-tile phase timestamps of CTA 0 (B2048_TC_DEBUG_CLOCK), else NULL
    // ---- fused rollout (policy_tc_kernel<true>): time-major rollout record, env state, env configuration
    uint64_t* ro_boards;      // [T + 1][n]
    uint8_t* ro_flags;        // [T + 1][n]
    uint8_t* ro_actions;      // [T][n]
    float* ro_rewards;        // [T][n]
    uint32_t* score;
    uint32_t* step;
    uint8_t* max_exp;
    int32_t* ep_len;          // nullable: run-to-termination bookkeeping (0 = running, else frozen)
    const uint8_t* tables;    // row tables + small tables (global memory; read through L1 / L2)
    const int32_t* slot_map;  // nullable: slot s of the launch is board slot_map[s] (run-to-termination rollouts launch
                              // the live boards only); n = number of slots, ro_stride = boards per record slice
    const int32_t* n_dev;     // nullable: the number of slots is read from device memory (b2048_compact_live wrote it),
                              // so the host can enqueue the next chunk without waiting for the count; n = upper bound
    int64_t ro_stride;
    uint64_t seed;
    int32_t t_begin, n_steps;
    uint32_t t0;
    b2048_env_cfg cfg;
};

// ------------------------------------------------------------------------------------------------ kernel
// Warp roles (21 warps = 672 threads, one CTA per SM):
//   warps 0..15  epilogue warps.  Warp w owns TMEM lanes / board rows 32*(w%4) .. +31 (the hardware's lane-quarter
//                rule) and, in every 64-column K slab of the next layer's operand, the 16 columns 16*(w/4) .. +15
//                (slab-major epilogues: all warps finish slab 0 first).
//   warp 16      issues every tcgen05.mma (lane 0), the weight-image bulk copies and owns TMEM alloc/dealloc.
//   warps 17..20 I/O warps, one thread per board: board load + A1 encode for the NEXT tile, and for the current tile
//                the 4 logits out of D3 -> mask load -> softmax -> Philox sample -> action store.  Global-memory
//                latency never sits on the MMA <-> epilogue critical path.
// Pipelining: the MMAs of K slab g are issued as soon as group g has written slab g (tensor core runs under the
// epilogues); A1 of tile i+1 is encoded right after epilogue 1 of tile i and MMA1(i+1) is issued as soon as layer 2
// of tile i has been issued, so it runs under epilogue 2(i).  All hand-offs are mbarriers (phase = tile parity).
constexpr int TC_H2_COL = 32;                                     // H2 (packed bf16 A operand of the head) inside the D2 region
constexpr int TC_EPI_THREADS = 512;
constexpr int TC_IO_THREADS = 128;
constexpr int TC_THREADS = TC_EPI_THREADS + 32 + TC_IO_THREADS;   // 16 epilogue warps + MMA warp + 4 I/O warps
constexpr int TC_ENV_GROUP = 128;                                 // fused rollout only: one env-step group = 4 warps
constexpr int TC_ENV_THREADS = 2 * TC_ENV_GROUP;                  // two groups, alternating over the CTA's tiles
constexpr int SM_ACT = SM_BAR + 256;                              // fused rollout only: 2 x 128 action bytes
constexpr int SM_TBL = SM_ACT + 256;                              // fused rollout only: small step tables
constexpr int SM_TOTAL_RO = SM_TBL + B2048_SMALL_BYTES;
static_assert(SM_TOTAL_RO <= 232448, "exceeds the 227 KB shared memory of an sm_100 CTA");

// Epilogue passes are SLAB-MAJOR: for every 64-column K slab s of the next layer's operand, warp (q, g) converts the 16
// accumulator columns 64 s + 16 g .. +15 of its 32 rows (ReLU -> bf16) and arrives on that slab's barrier.  All 16 warps finish
// slab 0 first, so the tensor core starts on the next layer after a quarter of the epilogue instead of after all of it.
// Epilogue 2 keeps H2 ON THE TENSOR CORE'S SIDE: bf16(relu(D2)) goes back into tensor memory as the packed A operand of the
// head MMAs (tcgen05.mma with A in TMEM: lane = row, one 32-bit column = two consecutive K elements) instead of into the A2
// shared-memory buffer.  A2 therefore belongs to layer 2 alone, and epilogue 1 of the NEXT item starts right after this pass
// instead of after the head MMAs.  Layout of the D2 region (256 columns): D3 = columns 0..15 (even K steps) + 16..31 (odd K
// steps; the sampler adds the two), H2 = columns 32..159 (slab s, warp group g: 32 + 32 s + 8 g .. +7), i.e. written IN PLACE
// over accumulator columns that belong to slabs <= s; columns 0..63 are drained before the first head MMA is issued.  Those columns are owned by other warps of the same lane quarter, so the four warps of a quarter meet at a
// named barrier once per slab, after their loads of that slab have landed and before anyone stores it.
// The same pass serves epilogue 1 (kDstCol = 0: H1 over the D1 region, the A operand of layer 2) — shared memory then holds
// weights and A1 only, and no generic-proxy -> async-proxy fence sits in either epilogue.
template <int kDstCol>
__device__ __forceinline__ void relu_store_tmem(uint32_t tlane_d2, int q, int g, int lane, uint32_t bar0) {
    static_assert(kDstCol >= 0 && kDstCol <= 32, "slab s must land in columns drained by slabs <= s");
    uint32_t r[2][16];
    tmem_ld16_issue(tlane_d2 + (uint32_t)(g * 16), r[0]);
    tmem_ld_wait(r[0]);
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        if (s + 1 < 4) tmem_ld16_issue(tlane_d2 + (uint32_t)((s + 1) * 64 + g * 16), r[(s + 1) & 1]);
        bar_sync(2 + q, 128);              // every warp of the quarter holds slab s in registers
        const uint32_t(&v)[16] = r[s & 1];
        uint32_t w[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) w[c] = relu_pack(v[2 * c], v[2 * c + 1]);
        tmem_st8(tlane_d2 + (uint32_t)(kDstCol + s * 32 + g * 8), w);
        tmem_st_wait();
        if (s + 1 < 4) tmem_ld_wait(r[(s + 1) & 1]);
        tc_fence_before();         // TMEM reads and writes ordered before the hand-off
        __syncwarp();
        if (lane == 0) mbar_arrive(bar0 + 8u * s);
    }
}

// kRollout = false: one policy step over all tiles (item = tile).
// kRollout = true : the whole rollout loop of b2048_rollout_many in ONE launch.  A CTA owns the tiles
//   first, first + grid, ... and walks the items (t, tile) for t = t_begin .. t_begin + n_steps - 1; boards are
//   independent, so no grid-wide synchronisation is needed.  The I/O thread that samples a board's action also plays
//   the env step for it (step_fast_rnd with the tables read through L1/L2, sharing the Philox block with the sampling
//   word) and writes slice t + 1 of the record — which the same thread reads back when the tile comes round again.
//   The MMA / epilogue warps see nothing but a longer item stream: weights, TMEM and barriers stay set up for the
//   whole rollout, and a step costs no launch, no image reload and no separate env kernel.
template <bool kRollout, bool kShaped = false>     // kShaped: the env configuration has reward-shaping terms (rollout only)
__global__ void __launch_bounds__(kRollout ? TC_THREADS + TC_ENV_THREADS : TC_THREADS, 1)
    policy_tc_kernel(const __grid_constant__ PolicyTcArgs args) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_BAR);
    const uint32_t bar_img = s_u32(&bars[0]), bar_a1 = s_u32(&bars[1]), bar_d1 = s_u32(&bars[2]), bar_d2 = s_u32(&bars[3]),
                   bar_d3 = s_u32(&bars[4]), bar_free = s_u32(&bars[5]);
    const uint32_t bar_slab0 = s_u32(&bars[6]);    // bars[6..9]   : A2 slab g written (layer-2 operand)
    const uint32_t bar_hslab0 = s_u32(&bars[10]);  // bars[10..13] : H2 slab g written (head operand)
    const uint32_t bar_act0 = s_u32(&bars[14]);    // [14..15] rollout: actions of env group g are in sAct[g]  (sampler -> env)
    const uint32_t bar_step0 = s_u32(&bars[16]);   // [16..17] rollout: env group g has written its item out    (env -> sampler)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM_BAR + 192);

    if (tid == 0) {
        mbar_init(bar_img, 1);
        mbar_init(bar_a1, 4);                       // one arrival per warp everywhere (elected lane after __syncwarp)
        mbar_init(bar_d1, 1);
        mbar_init(bar_d2, 1);
        mbar_init(bar_d3, 1);
        mbar_init(bar_free, TC_EPI_THREADS / 32 + TC_IO_THREADS / 32);
        for (int g = 0; g < 2; ++g) { mbar_init(bar_act0 + 8u * g, TC_IO_THREADS / 32); mbar_init(bar_step0 + 8u * g, TC_ENV_GROUP / 32); }
        for (int g = 0; g < 4; ++g) { mbar_init(bar_slab0 + 8u * g, TC_EPI_THREADS / 32); mbar_init(bar_hslab0 + 8u * g, TC_EPI_THREADS / 32); }
        mbar_init_fence();
    }
    // all 512 TMEM columns: D1 = 0..255, D2 = 256..511, D3 = 256..287 (two partial sums) and H2 (packed bf16) = 288..415 (over D2)
    const uint32_t tmem_base = tmem_setup(warp == 16, tmem_slot, 512u);
    const int64_t n_slots = (kRollout && args.n_dev) ? (int64_t)*args.n_dev : args.n;   // uniform over the grid
    const int64_t n_tiles = (n_slots + TC_M - 1) / TC_M;
    const int64_t first = blockIdx.x;
    // items of this CTA: its tiles, times the number of rollout steps
    const int n_owned = first < n_tiles ? (int)((n_tiles - first + gridDim.x - 1) / gridDim.x) : 0;
    const int n_items = kRollout ? n_owned * args.n_steps : n_owned;
    // With a single tile per CTA the next rollout item is the SAME boards one step later: its A1 can only be encoded
    // after this item's env step, so layer 1 of the next item is issued after this item's head instead of before it.
    const bool prefetch = !kRollout || n_owned > 1;

    if (warp == 16) {
        // ============================ MMA / copy warp ============================
        // All 32 lanes walk the loops CONVERGENTLY (item / slab counters, barrier probes and the 32-bit descriptor words live in
        // uniform registers); lane 0 only issues the asynchronous instructions — no ELECT / R2UR waterfall and no BRA.U.ANY loop
        // per tcgen05.mma as under `if (lane == 0) { whole loop }`.  Measured: the item period does not change, i.e. the ~130
        // cycles every head MMA costs are NOT issue overhead either (nor the accumulate dependency, nor the A operand's source):
        // the tensor pipe has a per-instruction floor of that size on this part, which a full-width M128 N256 K16 MMA (128
        // cycles of math) hides and an M128 N16 K16 one (8 cycles) does not (DESIGN.md, K3).
        const bool leader = lane == 0;
        const uint32_t lA1 = dlo_ns(s_u32(smem + SM_A1)), lW1 = dlo_ns(s_u32(smem + IMG_W1));
        const uint32_t lW2 = dlo_sw(s_u32(smem + IMG_W2)), lW3 = dlo_sw(s_u32(smem + IMG_W3));
        const uint32_t lBias = dlo_ns(s_u32(smem + IMG_BIAS));
        const uint32_t lOnes1 = dlo_ns(s_u32(smem + IMG_ONES1)), lOnes2 = dlo_ns(s_u32(smem + IMG_ONES2));
        if (leader) {
            mbar_expect_tx(bar_img, (uint32_t)IMG_BYTES);
            bulk_load_chunked<16384u>(s_u32(smem), args.img, (uint32_t)IMG_BYTES, bar_img);
        }
        __syncwarp();
        mbar_wait(bar_img, 0);
        auto issue_layer1 = [&](uint32_t ph) {   // D1 = A1 . W1^T + b1   (called by the whole warp)
            mbar_wait(bar_a1, ph);
            tc_fence_after();
            if (leader) {
                umma_w(tmem_base, lA1, DH_NOSW, lW1, DH_NOSW, kIdesc, 0u);
                umma_w(tmem_base, lOnes1, DH_ONES, lBias, DH_NOSW, kIdesc, 1u);
                umma_commit(bar_d1);
            }
        };
        uint32_t ph = 0;
        if (n_items > 0) issue_layer1(0u);
        for (int item = 0; item < n_items; ++item) {
            if (!prefetch && item != 0) issue_layer1(ph);
            const bool mdbg = args.debug_clock != nullptr && blockIdx.x == 0 && item < 4 && leader;
            // ---- layer 2, slab by slab as epilogue 1 produces them: A = H1 in tensor memory (D1 region, 8 columns per K = 16
            //      step), B = the W2 slab in shared memory (descriptor low word + 2 per 32-byte K step, + 2048 per slab)
            for (uint32_t g = 0; g < 4; ++g) {
                mbar_wait(bar_slab0 + 8u * g, ph);
                if (g == 0 && item != 0) mbar_wait(bar_free, ph ^ 1u);       // D2/D3 drained by the previous tile
                if (g == 0 && mdbg) args.debug_clock[64 + 4 * item] = clock64();
                tc_fence_after();
                const uint32_t a0 = tmem_base + g * 32u, b0 = lW2 + g * 2048u;
                if (leader) {
                    umma_w_ts(tmem_base + 256u, a0, b0, DH_SW, kIdesc, g ? 1u : 0u);
                    umma_w_ts(tmem_base + 256u, a0 + 8u, b0 + 2u, DH_SW, kIdesc, 1u);
                    umma_w_ts(tmem_base + 256u, a0 + 16u, b0 + 4u, DH_SW, kIdesc, 1u);
                    umma_w_ts(tmem_base + 256u, a0 + 24u, b0 + 6u, DH_SW, kIdesc, 1u);
                }
            }
            if (leader) {
                umma_w(tmem_base + 256u, lOnes2, DH_ONES, lBias, DH_NOSW, kIdesc, 1u);           // + b2
                umma_commit(bar_d2);
            }
            // ---- next tile's layer 1 runs under this tile's epilogue 2 — as soon as its A1 is there AND this item's layer 2 has
            //      completed (it overwrites the D1 region layer 2 reads H1 from; bar_d2, the phase the epilogue warps wait for too).
            //      Both are probed, not waited for, until the head has been issued: the logits feed the sampler, the env step
            //      and, through bar_free, the next item's layer 2.
            bool l1_pending = prefetch && item + 1 < n_items;
            auto try_layer1 = [&]() {
                if (l1_pending && mbar_test(bar_d2, ph) && mbar_test(bar_a1, ph ^ 1u)) { issue_layer1(ph ^ 1u); l1_pending = false; }
            };
            // ---- head: D3 = H2 . W3^T, slab by slab as epilogue 2 produces them; A = H2 in tensor memory (D2 region, from
            //      column TC_H2_COL).  D3 = D2 columns 0..31 (two partial sums, even / odd K steps), which belong to slab 0 and
            //      have been drained by every warp before hslab[0] completes.
            for (uint32_t g = 0; g < 4; ++g) {
                try_layer1();
                while (!mbar_test(bar_hslab0 + 8u * g, ph)) try_layer1();
                if (mdbg && g == 3) args.debug_clock[64 + 4 * item + 1] = clock64();
                tc_fence_after();
                const uint32_t a0 = tmem_base + 256u + (uint32_t)TC_H2_COL + g * 32u, b0 = lW3 + g * 128u;
                if (leader) {
                    umma_w_ts(tmem_base + 256u, a0, b0, DH_SW, kIdescHead, g ? 1u : 0u);
                    umma_w_ts(tmem_base + 256u + 16u, a0 + 8u, b0 + 2u, DH_SW, kIdescHead, g ? 1u : 0u);
                    umma_w_ts(tmem_base + 256u, a0 + 16u, b0 + 4u, DH_SW, kIdescHead, 1u);
                    umma_w_ts(tmem_base + 256u + 16u, a0 + 24u, b0 + 6u, DH_SW, kIdescHead, 1u);
                }
            }
            if (leader) umma_commit(bar_d3);
            if (mdbg) args.debug_clock[64 + 4 * item + 2] = clock64();
            if (l1_pending) { mbar_wait(bar_d2, ph); issue_layer1(ph ^ 1u); }
            ph ^= 1u;
        }
        __syncwarp();
    } else if (warp < 16) {
        // ============================ epilogue warps ============================
        const int q = warp & 3, g = warp >> 2;
        const int row = q * 32 + lane;                                          // board row inside the tile = TMEM lane
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t ph = 0;
        for (int item = 0; item < n_items; ++item) {
            const bool dbg = args.debug_clock != nullptr && blockIdx.x == 0 && tid == 0 && item < 8;
            long long* dc = dbg ? args.debug_clock + 8 * item : nullptr;
            if (dbg) dc[0] = clock64();
            // ---- epilogue 1: H1 = bf16(relu(D1)), slab by slab, packed in place over the D1 region (columns 0..127): the A
            //      operand of layer 2 in tensor memory
            mbar_wait(bar_d1, ph);
            if (dbg) dc[1] = clock64();
            tc_fence_after();
            relu_store_tmem<0>(tlane, q, g, lane, bar_slab0);
            if (dbg) dc[2] = clock64();
            // ---- epilogue 2: H2 = bf16(relu(D2)), slab by slab, packed back into tensor memory (relu_store_tmem)
            mbar_wait(bar_d2, ph);
            if (dbg) dc[3] = clock64();
            tc_fence_after();
            relu_store_tmem<TC_H2_COL>(tlane + 256u, q, g, lane, bar_hslab0);
            if (args.debug_clock != nullptr && blockIdx.x == 0 && item < 4 && lane == 0)    // the slowest warp's end of epilogue 2
                atomicMax(reinterpret_cast<unsigned long long*>(args.debug_clock) + 80 + item, (unsigned long long)clock64());
            if (lane == 0) mbar_arrive(bar_free);      // this warp's D2 reads were fenced before its hslab arrivals
            if (dbg) dc[4] = clock64();
            ph ^= 1u;
        }
    } else {
        // ============================ I/O warps (17..20), one thread per board ============================
        // They keep every global-memory latency (board loads, mask loads, action stores) and the softmax / Philox
        // sampling off the MMA <-> epilogue critical path: encode A1 of tile i+1 while tile i is in flight, then pick
        // up the 4 logits of tile i from D3.
        const int q = warp & 3;                                                 // TMEM lane quarter this warp may read
        const int row = q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        const float* sB3 = reinterpret_cast<const float*>(smem + IMG_B3);
        uint32_t ph = 0;

        // An item is (j, r): the CTA's j-th tile in rollout round r (plain policy step: r = 0 throughout).  The pair is
        // advanced incrementally — these warps run long dependent chains alone on their schedulers, and an integer
        // division by n_owned costs them more than the softmax.
        auto tile_of = [&](int j) -> int64_t { return first + (int64_t)j * gridDim.x; };
        auto slice_of = [&](int r) -> int64_t { return kRollout ? (int64_t)args.t_begin + r : 0; };
        uint8_t* sAct = smem + SM_ACT;                                          // rollout: sampled actions of the item

        if (warp < 21) {
            // ---------------- sampler warps (17..20): A1 encode, D3 -> softmax -> action ----------------
            const uint64_t* board_base = kRollout ? args.ro_boards : args.board;
            const uint8_t* mask_base = kRollout ? args.ro_flags : args.mask_flags;
            // Rollout: tile j of the CTA (item % n_owned) belongs to env group j & 1, so a board is always stepped by
            // the same thread.  Group g's ord-th item is item_of(g, ord); bar_step[g] completes once per item of the
            // group, in order, and the sampler waits for every phase exactly once, in order.  The boards / flags
            // of an item are written by the same group one round (n_owned items, cnt[g] group items) earlier.
            int steps_waited[2] = {0, 0};
            auto wait_steps_through = [&](int g, int ord) {
                while (steps_waited[g] <= ord) {
                    mbar_wait(bar_step0 + 8u * g, (uint32_t)steps_waited[g] & 1u);
                    ++steps_waited[g];
                }
            };
            auto ord_of = [&](int j, int r) {   // ordinal of item (j, r) among the items of its group j & 1
                return r * ((n_owned + 1 - (j & 1)) >> 1) + (j >> 1);
            };
            auto wait_inputs_of = [&](int j, int r) {   // written by the same group one round earlier
                if (r > 0) wait_steps_through(j & 1, ord_of(j, r - 1));
            };

            auto encode_a1 = [&](int j, int r) {   // this thread's board -> 16 bf16 in the A1 core matrices
                const int64_t s = tile_of(j) * TC_M + row;
                uint64_t bd = 0ull;
                if (s < n_slots) {
                    const int64_t b = (kRollout && args.slot_map) ? args.slot_map[s] : s;
                    bd = board_base[slice_of(r) * (kRollout ? args.ro_stride : args.n) + b];
                }
                uint32_t packed[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    uint32_t e0 = (uint32_t)(bd >> (8 * j)) & 0xFu, e1 = (uint32_t)(bd >> (8 * j + 4)) & 0xFu;
                    float v0, v1;
                    if (args.obs_mode == B2048_OBS_RAW) { v0 = e0 ? (float)(1u << e0) : 0.0f; v1 = e1 ? (float)(1u << e1) : 0.0f; }
                    else { v0 = (float)e0 * args.obs_scale; v1 = (float)e1 * args.obs_scale; }
                    __nv_bfloat162 p = __floats2bfloat162_rn(v0, v1);
                    packed[j] = *reinterpret_cast<uint32_t*>(&p);
                }
                uint8_t* a1 = smem + SM_A1 + (row >> 3) * 256 + (row & 7) * 16;
                *reinterpret_cast<uint4*>(a1) = make_uint4(packed[0], packed[1], packed[2], packed[3]);
                *reinterpret_cast<uint4*>(a1 + 128) = make_uint4(packed[4], packed[5], packed[6], packed[7]);
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_a1);
            };

            if (n_items > 0) encode_a1(0, 0);
            mbar_wait(bar_img, 0);                                              // b3 lives in the image
            int j = 0, r = 0;
            for (int item = 0; item < n_items; ++item) {
                int jn = j + 1, rn = r;                                          // the next item
                if (jn == n_owned) { jn = 0; ++rn; }
                const int64_t s = tile_of(j) * TC_M + row;
                const int64_t slice = slice_of(r);
                const bool valid = s < n_slots;
                const int64_t b = (kRollout && valid && args.slot_map) ? args.slot_map[s] : s;   // board behind the slot
                const int64_t stride = kRollout ? args.ro_stride : args.n;
                const bool use_mask = args.mask_flags != nullptr;               // rollout: non-NULL iff the policy is masked
                if (kRollout) wait_inputs_of(j, r);
                uint32_t fl = 0xFu;
                if (valid && use_mask) fl = mask_base[slice * stride + b];      // requested early, used after D3
                const uint32_t t_env = kRollout ? args.t0 + (uint32_t)slice + 1u : args.t;
                uint32_t w3 = 0u;
                if (valid && !args.greedy && (kRollout || args.action))
                    w3 = stream_keyed(args.keys, args.gid0 + (uint64_t)b, t_env, B2048_DOM_STEP).w3;
                // A1 is free once this item's layer-1 MMAs have completed
                mbar_wait(bar_d1, ph);
                if (prefetch && item + 1 < n_items) {
                    if (kRollout) wait_inputs_of(jn, rn);
                    encode_a1(jn, rn);
                }
                const bool dbg = args.debug_clock != nullptr && blockIdx.x == 0 && tid == TC_EPI_THREADS + 32 && item < 8;
                if (dbg && item < 4) args.debug_clock[64 + 4 * item + 3] = clock64();
                mbar_wait(bar_d3, ph);
                if (dbg) args.debug_clock[8 * item + 5] = clock64();
                tc_fence_after();
                uint32_t r4[4], r4b[4];
                tmem_ld4_issue(tlane + 256u, r4);
                tmem_ld4_issue(tlane + 256u + 16u, r4b);
                tmem_ld_wait(r4);                              // waits for both loads
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_free);
                const float lg0 = (__uint_as_float(r4[0]) + __uint_as_float(r4b[0])) + sB3[0];
                const float lg1 = (__uint_as_float(r4[1]) + __uint_as_float(r4b[1])) + sB3[1];
                const float lg2 = (__uint_as_float(r4[2]) + __uint_as_float(r4b[2])) + sB3[2];
                const float lg3 = (__uint_as_float(r4[3]) + __uint_as_float(r4b[3])) + sB3[3];
                uint32_t a = 0;
                if (valid) {
                    float m0 = (use_mask && !(fl & 1u)) ? -1e9f : lg0, m1 = (use_mask && !(fl & 2u)) ? -1e9f : lg1;
                    float m2 = (use_mask && !(fl & 4u)) ? -1e9f : lg2, m3 = (use_mask && !(fl & 8u)) ? -1e9f : lg3;
                    // fast-math softmax (ex2.approx / rcp.approx, ~2^-21 relative): this thread is on the rollout's
                    // critical path and the bf16 logits carry 2^-9 anyway
                    float mx = fmaxf(fmaxf(m0, m1), fmaxf(m2, m3));
                    float e0 = __expf(m0 - mx), e1 = __expf(m1 - mx), e2 = __expf(m2 - mx), e3 = __expf(m3 - mx);
                    float inv = __fdividef(1.0f, e0 + e1 + e2 + e3);
                    float p0 = e0 * inv, p1 = e1 * inv, p2 = e2 * inv, p3 = e3 * inv;
                    if (!kRollout && args.probs) *reinterpret_cast<float4*>(args.probs + s * 4) = make_float4(p0, p1, p2, p3);
                    if (!kRollout && args.logits) *reinterpret_cast<float4*>(args.logits + s * 4) = make_float4(lg0, lg1, lg2, lg3);
                    if (!kRollout && args.head_out) {
                        const float lg[4] = {lg0, lg1, lg2, lg3};
                        for (int k = 0; k < args.n_out; ++k) args.head_out[s * args.n_out + k] = lg[k];
                    }
                    if (kRollout || args.action) {
                        if (args.greedy) {
                            float q0 = (!use_mask || (fl & 1u)) ? p0 : 0.0f, q1 = (!use_mask || (fl & 2u)) ? p1 : 0.0f;
                            float q2 = (!use_mask || (fl & 4u)) ? p2 : 0.0f, q3 = (!use_mask || (fl & 8u)) ? p3 : 0.0f;
                            a = 0; float best = q0;
                            if (q1 > best) { best = q1; a = 1; }
                            if (q2 > best) { best = q2; a = 2; }
                            if (q3 > best) { best = q3; a = 3; }
                        } else {
                            float c0 = p0, c1 = c0 + p1, c2 = c1 + p2, c3 = c2 + p3;
                            float u = ((float)(w3 >> 8) + 0.5f) * (1.0f / 16777216.0f) * c3;
                            a = (u >= c0 ? 1u : 0u) + (u >= c1 ? 1u : 0u) + (u >= c2 ? 1u : 0u);
                            float pa = a == 0 ? p0 : a == 1 ? p1 : a == 2 ? p2 : p3;
                            if (!(pa > 0.0f)) {
                                if (p3 > 0.0f) a = 3;
                                if (p2 > 0.0f) a = 2;
                                if (p1 > 0.0f) a = 1;
                                if (p0 > 0.0f) a = 0;
                            }
                        }
                        if (kRollout) args.ro_actions[slice * stride + b] = (uint8_t)a;
                        else args.action[s] = (uint8_t)a;
                    }
                }
                if (kRollout) {
                    // hand the actions to the item's env group (one slot per group: its previous item must be finished)
                    const int g = j & 1, ord = ord_of(j, r);
                    wait_steps_through(g, ord - 1);
                    sAct[g * TC_M + row] = (uint8_t)a;
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_act0 + 8u * g);
                    if (dbg) args.debug_clock[8 * item + 6] = clock64();
                    if (!prefetch && item + 1 < n_items) {
                        wait_inputs_of(jn, rn);
                        encode_a1(jn, rn);
                    }
                }
                j = jn; r = rn;
                ph ^= 1u;
            }
        } else if (kRollout) {
            // ---------------- env warps (21..28): one thread per board plays the sampled action ----------------
            // Two groups of four warps; group g owns the CTA's tiles j with j & 1 == g.  One warp per scheduler running
            // the ~700-instruction step chain is latency-bound (about 6 K cycles per item, more than the 5 K the tensor
            // pipeline needs), so the groups alternate and each has two item periods per step.
            // Same contract as step_fast_kernel (b2048_env.cu); the row tables are read through L1 / L2 (shared memory
            // is full of weights).  Everything a board's env thread reads back next time (board, flags, counters,
            // episode length) it wrote itself; the sampler warps see the new slice through bar_step.
            // The small tables (per-action selectors, merge statistics: 2.2 KB) are copied into shared memory so that
            // the only L2 round trip on a step's dependency chain is the row lookup itself.
            {
                const uint4* src = reinterpret_cast<const uint4*>(args.tables + B2048_LUT_BYTES);
                uint4* dst = reinterpret_cast<uint4*>(smem + SM_TBL);
                for (int i = tid - TC_THREADS; i < B2048_SMALL_BYTES / 16; i += TC_ENV_THREADS) dst[i] = src[i];
                bar_sync(1, TC_ENV_THREADS);
            }
            const int grp = (warp - 21) >> 2;
            const uint32_t bar_act = bar_act0 + 8u * grp, bar_step = bar_step0 + 8u * grp;
            // this group's items: tiles grp, grp + 2, ... of every round
            FastTables T;
            T.left = reinterpret_cast<const uint16_t*>(args.tables);
            T.merge = args.tables + B2048_LUT_LEFT_BYTES;
            T.agg = reinterpret_cast<const AggEntry*>(smem + SM_TBL + B2048_SMALL_AGG_OFF);
            T.sel = reinterpret_cast<const SelEntry*>(smem + SM_TBL + B2048_SMALL_SEL_OFF);
            T.act = smem + SM_TBL + B2048_SMALL_ACT_OFF;

            struct EnvIn { uint64_t bd; uint32_t score, step, max_exp, fin; int32_t ep; };
            auto load_in = [&](int j, int r) {
                EnvIn e = {0ull, 0u, 0u, 2u, 0u, 0};
                const int64_t s = tile_of(j) * TC_M + row;
                if (s < n_slots) {
                    const int64_t b = args.slot_map ? args.slot_map[s] : s;
                    const int64_t i = slice_of(r) * args.ro_stride + b;
                    e.bd = args.ro_boards[i]; e.fin = args.ro_flags[i];
                    e.score = args.score[b]; e.step = args.step[b]; e.max_exp = args.max_exp[b];
                    if (args.ep_len) e.ep = args.ep_len[b];
                }
                return e;
            };
            const int own_tiles = (n_owned + 1 - grp) >> 1;   // tiles of this group per round
            const int n_rounds = n_owned > 0 ? n_items / n_owned : 0;
            int j = grp, r = own_tiles > 0 ? 0 : n_rounds;
            EnvIn cur = r < n_rounds ? load_in(j, r) : EnvIn{0ull, 0u, 0u, 2u, 0u, 0};
            while (r < n_rounds) {
                int jn = j + 2, rn = r;                                          // the group's next item
                if (jn >= n_owned) { jn = grp; ++rn; }
                const int item = r * n_owned + j;
                const int64_t s = tile_of(j) * TC_M + row;
                const int64_t slice = slice_of(r);
                const bool valid = s < n_slots;
                const int64_t b = (valid && args.slot_map) ? args.slot_map[s] : s;
                const uint32_t t_env = args.t0 + (uint32_t)slice + 1u;
                FastIO io;
                io.lo = (uint32_t)cur.bd; io.hi = (uint32_t)(cur.bd >> 32);
                io.score = cur.score; io.step = cur.step; io.max_exp = cur.max_exp; io.mask_in = 0u;
                const uint32_t fin = cur.fin;
                const bool frozen = cur.ep != 0;
                Rand4 rr = Rand4{0u, 0u, 0u, 0u};
                if (valid && !frozen) rr = stream_keyed(args.keys, args.gid0 + (uint64_t)b, t_env, B2048_DOM_STEP);
                // Next item's inputs: with several tiles per CTA this thread wrote them at least one item ago, so the
                // loads go out now and land under this item's step; with one tile they are this step's outputs.
                EnvIn nxt = cur;
                if (own_tiles > 1 && rn < n_rounds) nxt = load_in(jn, rn);
                mbar_wait(bar_act, ph);
                const bool dbg = args.debug_clock != nullptr && blockIdx.x == 0 && (tid - TC_THREADS) % TC_ENV_GROUP == 0 && item < 8;
                if (dbg) args.debug_clock[8 * item + 7] = clock64();
                if (valid) {
                    const int64_t o = (slice + 1) * args.ro_stride + b;
                    if (frozen) {
                        args.ro_boards[o] = cur.bd;
                        args.ro_rewards[slice * args.ro_stride + b] = 0.0f;
                        io.flags = fin & ~B2048_F_CHANGED;
                        args.ro_flags[o] = (uint8_t)io.flags;
                    } else {
                        io.action = sAct[grp * TC_M + row];
                        step_fast_rnd<B2048_ACT_BUFFER, true, kShaped>(io, args.cfg, rr, args.keys, args.gid0 + (uint64_t)b, t_env, T);
                        if (args.ep_len && (io.flags & (B2048_F_DONE | B2048_F_TRUNC))) {
                            args.ep_len[b] = (int32_t)(slice + 1);
                            cur.ep = (int32_t)(slice + 1);
                        }
                        args.ro_boards[o] = (uint64_t)io.lo | ((uint64_t)io.hi << 32);
                        args.score[b] = io.score; args.step[b] = io.step; args.max_exp[b] = (uint8_t)io.max_exp;
                        args.ro_rewards[slice * args.ro_stride + b] = io.reward;
                        args.ro_flags[o] = (uint8_t)io.flags;
                    }
                }
                if (own_tiles == 1) {   // same boards next time: carry the state in registers
                    nxt.bd = (uint64_t)io.lo | ((uint64_t)io.hi << 32);
                    nxt.score = io.score; nxt.step = io.step; nxt.max_exp = io.max_exp; nxt.fin = io.flags; nxt.ep = cur.ep;
                }
                cur = nxt;
                j = jn; r = rn;
                __threadfence_block();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_step);
                ph ^= 1u;
            }
        }
    }

    tmem_teardown(warp == 16, tmem_base, 512u);
}

// Builds the bf16 weight image of a 16 -> 256 -> 256 -> n_out (n_out <= 4) network into `img` (IMG_BYTES, device).
void launch_tc_prepare(const b2048_mlp_desc* mlp, uint8_t* img, cudaStream_t stream) {
    policy_tc_prepare_kernel<<<64, 256, 0, stream>>>(mlp->W[0], mlp->b[0], mlp->W[1], mlp->b[1], mlp->W[2], mlp->b[2],
                                                      mlp->dims[3], img);
}

// Allocates the handle's weight-image buffer (shared by the policy, rollout and training kernels) and opts the kernels of
// this file into their dynamic shared memory sizes.
int ensure_tc_image(b2048_handle* h) {
    if (!h->tc_image) {
        cudaError_t e = cudaMalloc(&h->tc_image, IMG_BYTES);
        if (e != cudaSuccess) return check_cuda(e, "cudaMalloc(tc_image)");
    }
    if (!(h->attrs & ATTR_POLICY_TC)) {
        cudaError_t e = cudaFuncSetAttribute(policy_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL2);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(policy_tc_kernel)");
        e = cudaFuncSetAttribute(policy_tc_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL_RO);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(policy_tc_kernel<rollout>)");
        e = cudaFuncSetAttribute(policy_tc_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SM_TOTAL_RO);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(policy_tc_kernel<rollout, shaped>)");
        h->attrs |= ATTR_POLICY_TC;
    }
    return B2048_OK;
}

static int print_debug_clock(const b2048_handle* h, cudaStream_t stream) {
    long long hbuf[96];
    { int st = debug_clock_read(h, hbuf, 96, stream); if (st != B2048_OK) return st; }
    for (int k = 0; k < 6; ++k)
        fprintf(stderr,
                "[tc clock] item %d: wait_d1+d3 %lld epi1 %lld wait_d2 %lld epi2 %lld | total %lld | to next %lld | io: d3 seen +%lld, "
                "sample %lld | env: actions seen +%lld\n",
                k, hbuf[8 * k + 1] - hbuf[8 * k], hbuf[8 * k + 2] - hbuf[8 * k + 1], hbuf[8 * k + 3] - hbuf[8 * k + 2],
                hbuf[8 * k + 4] - hbuf[8 * k + 3], hbuf[8 * k + 4] - hbuf[8 * k], hbuf[8 * k + 8] - hbuf[8 * k],
                hbuf[8 * k + 5] - hbuf[8 * k], hbuf[8 * k + 6] - hbuf[8 * k + 5], hbuf[8 * k + 7] - hbuf[8 * k]);
    for (int k = 0; k < 4; ++k)      // MMA warp / sampler, relative to the item's start (epilogue warps' clock 0)
        fprintf(stderr, "[tc clock] item %d: mma: layer 2 starts +%lld, last H2 slab seen +%lld, d3 committed +%lld | sampler waits for d3 from +%lld\n",
                k, hbuf[64 + 4 * k] - hbuf[8 * k], hbuf[64 + 4 * k + 1] - hbuf[8 * k], hbuf[64 + 4 * k + 2] - hbuf[8 * k],
                hbuf[64 + 4 * k + 3] - hbuf[8 * k]);
    for (int k = 0; k < 4; ++k) fprintf(stderr, "[tc clock] item %d: slowest epilogue warp leaves epilogue 2 at +%lld\n", k, hbuf[80 + k] - hbuf[8 * k]);
    return B2048_OK;
}

int launch_policy_tc(b2048_handle* h, const b2048_mlp_desc* mlp, const uint64_t* board, const uint8_t* mask_flags,
                     uint8_t* action, float* probs, float* logits, int64_t n, uint64_t seed, uint64_t gid0, uint32_t t,
                     int greedy, cudaStream_t stream, bool rebuild_image) {
    if (!fixed_tc_net(mlp) || mlp->dims[3] != 4 || h->smem_optin < SM_TOTAL2) return B2048_ERR_UNSUPPORTED;
    { int st = ensure_tc_image(h); if (st != B2048_OK) return st; }
    // The image is rebuilt on every stand-alone call (71 K parameters): the library never caches weights across
    // calls.  b2048_rollout_many builds it once for the whole loop (parameters cannot change inside one call).
    if (rebuild_image) launch_tc_prepare(mlp, h->tc_image, stream);
    PolicyTcArgs a{};
    a.img = h->tc_image; a.board = board; a.mask_flags = mask_flags; a.action = action; a.probs = probs; a.logits = logits;
    a.n_out = 4; a.n = n; a.keys = make_keys(seed); a.gid0 = gid0; a.t = t; a.greedy = greedy; a.obs_mode = mlp->obs_mode;
    a.obs_scale = mlp->obs_log2_scale; a.seed = seed; a.n_steps = 1; a.ro_stride = n;
    a.debug_clock = debug_clock_begin(h, B2048_DBG_TC_CLOCKS, stream);
    int64_t tiles = (n + TC_M - 1) / TC_M;
    int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
    policy_tc_kernel<false><<<grid, TC_THREADS, SM_TOTAL2, stream>>>(a);
    int st = check_cuda(cudaGetLastError(), "policy_tc_kernel launch");
    if (st == B2048_OK && a.debug_clock) st = print_debug_clock(h, stream);
    return st;
}

// b2048_mlp_forward on the tensor cores: out[n][n_out] = head outputs of a 16-256-256-n_out (n_out <= 4) ReLU network
// (the critic's V(s) for the TD targets, reinforce_agent.py:425-437).
int launch_forward_tc(b2048_handle* h, const b2048_mlp_desc* mlp, const uint64_t* board, float* out, int64_t n,
                      cudaStream_t stream) {
    if (!fixed_tc_net(mlp) || h->smem_optin < SM_TOTAL2 || n < 4096) return B2048_ERR_UNSUPPORTED;
    { int st = ensure_tc_image(h); if (st != B2048_OK) return st; }
    launch_tc_prepare(mlp, h->tc_image, stream);
    PolicyTcArgs a{};
    a.img = h->tc_image; a.board = board; a.head_out = out; a.n_out = mlp->dims[3]; a.n = n; a.keys = make_keys(0); a.greedy = 1;
    a.obs_mode = mlp->obs_mode; a.obs_scale = mlp->obs_log2_scale; a.n_steps = 1; a.ro_stride = n;
    int64_t tiles = (n + TC_M - 1) / TC_M;
    int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
    policy_tc_kernel<false><<<grid, TC_THREADS, SM_TOTAL2, stream>>>(a);
    return check_cuda(cudaGetLastError(), "policy_tc_kernel (forward) launch");
}

// The whole rollout loop of b2048_rollout_many in one launch (policy_tc_kernel<true>).  When the network / env
// configuration is outside what the fused kernel implements, the caller runs the two-kernels-per-step loop.
int launch_rollout_tc(b2048_handle* h, const b2048_mlp_desc* mlp, uint64_t* boards, uint8_t* flags, uint8_t* actions,
                      float* rewards, uint32_t* score, uint32_t* step, uint8_t* max_exp, int32_t* ep_len,
                      const b2048_env_cfg* cfg, int64_t B, int32_t t_begin, int32_t n_steps, uint64_t seed, uint64_t gid0,
                      uint32_t t0, int use_mask, int greedy, const int32_t* slot_map, int64_t n_slots, const int32_t* n_slots_dev,
                      cudaStream_t stream) {
    const bool net_ok = fixed_tc_net(mlp) && mlp->dims[3] == 4 && h->smem_optin >= SM_TOTAL_RO;
    // every action-mask-on reward configuration (step_fast_rnd carries the shaping terms; the counters are always tracked here)
    const bool env_ok = score && step && max_exp && cfg->use_action_mask &&
                        (cfg->reward_mode == B2048_REWARD_SUM || cfg->reward_mode == B2048_REWARD_LOG2);
    // slot_map: only the listed boards are played (n_slots of them); without it all B boards
    const int64_t n = slot_map ? n_slots : B;
    const int64_t tiles = (n + TC_M - 1) / TC_M;
    if (!net_ok || !env_ok || B < 4096 || tiles * (int64_t)n_steps > 0x7FFFFFFF || (h->debug & (1u << B2048_DBG_NO_FUSED_ROLLOUT)))
        return B2048_ERR_UNSUPPORTED;
    if (n == 0) return B2048_OK;
    { int st = ensure_tc_image(h); if (st != B2048_OK) return st; }
    launch_tc_prepare(mlp, h->tc_image, stream);
    PolicyTcArgs a{};
    a.img = h->tc_image; a.mask_flags = use_mask ? flags : nullptr; a.n_out = 4; a.n = n; a.keys = make_keys(seed); a.gid0 = gid0;
    a.greedy = greedy; a.obs_mode = mlp->obs_mode; a.obs_scale = mlp->obs_log2_scale;
    a.ro_boards = boards; a.ro_flags = flags; a.ro_actions = actions; a.ro_rewards = rewards; a.score = score; a.step = step;
    a.max_exp = max_exp; a.ep_len = ep_len; a.tables = h->d_tables; a.seed = seed; a.t_begin = t_begin; a.n_steps = n_steps;
    a.t0 = t0; a.cfg = *cfg; a.cfg.action_mode = B2048_ACT_BUFFER; a.slot_map = slot_map; a.n_dev = slot_map ? n_slots_dev : nullptr;
    a.ro_stride = B;
    int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
    a.debug_clock = debug_clock_begin(h, B2048_DBG_TC_CLOCKS, stream);
    if (cfg_is_shaped(*cfg)) policy_tc_kernel<true, true><<<grid, TC_THREADS + TC_ENV_THREADS, SM_TOTAL_RO, stream>>>(a);
    else policy_tc_kernel<true, false><<<grid, TC_THREADS + TC_ENV_THREADS, SM_TOTAL_RO, stream>>>(a);
    int st = check_cuda(cudaGetLastError(), "policy_tc_kernel<rollout> launch");
    if (st == B2048_OK && a.debug_clock) st = print_debug_clock(h, stream);
    return st;
}

}  // namespace b2
