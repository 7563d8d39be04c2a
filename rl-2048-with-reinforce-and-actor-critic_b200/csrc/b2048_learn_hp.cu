// b2048_learn_hp.cu — K6 on the tensor cores at float32-grade accuracy (precision 3, what "auto" selects).
//
// Why: the gradient of update_batch (src/reinforce_agent.py:403-555, _backpropagation :639-678) is a heavily cancelling
// sum over samples, and a ReLU unit whose pre-activation is within the forward pass's rounding error of zero switches
// on / off relative to the float32 arithmetic of the reference.  The relative error of the summed gradient therefore
// scales with the SQUARE ROOT of the forward rounding error (measured on rollout-derived batches: bf16 operands 5 %,
// fp16 1.5 %, float32 itself 0.06 % against float64).  Single-bf16 tensor-core arithmetic (b2048_learn_tc.cu) cannot
// meet the 1e-2 parity bar; this path does:
//
//  fwd_hp_kernel   forward pass with every operand split into fp16 hi + lo (x = hi + lo to 22 bits) and three
//                  tcgen05.mma per product (hi.hi + lo.hi + hi.lo, fp32 accumulation in TMEM): pre-activations accurate
//                  to ~1e-6 relative.  The 256 KB of split W2 do not fit in shared memory next to the activations, so
//                  the weights STREAM through a 3-slot ring of 32 KB K-slab units (bulk async copies from the L2-resident
//                  image), and the split activations go through a 2-stage ring that the epilogues fill slab by slab.
//                  Outputs: head outputs (logits / V), the ReLU masks of both layers (64 bits per thread, bit-packed),
//                  and the fp16 activation images H1, H2 for the dW GEMMs.
//  bwd_tc_kernel   backward deltas only (no forward): d3 from the float32 logits, D5 = d3 W3^T, DL2 = D5 . mask2,
//                  D4 = DL2 W2 (the resident fp16 W2 image read MN-major), DL1 = D4 . mask1, fp16 operands with a
//                  power-of-two loss scale (the coefficients are ~1e-8).  Rounding the backward operands perturbs the
//                  gradient linearly (no mask flips): 0.04 % at fp16.
//  atb_tc_kernel   (b2048_learn_tc.cu) the dW GEMMs on the fp16 images, un-scaled on the way out.
//  bwd_tc_ent_kernel / update_pipe_ent_kernel   bwd_tc_kernel / update_pipe_kernel with the entropy bonus in the policy head's
//                  delta (b2048_mlp_backward_entropy, b2048_entropy.cuh)
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <ctime>
#include <type_traits>
#include <unistd.h>

#include "b2048_device.cuh"
#include "b2048_entropy.cuh"
#include "b2048_internal.h"
#include "b2048_tc.cuh"
#include "b2048_learn_tc.cuh"

namespace b2 {

// ------------------------------------------------------------------------------------------------ split-weight image
constexpr int HP_UNIT = 32768;                  // one streamed unit: a 64-wide K slab of W2 hi or lo, [256 rows x 128 B]
constexpr int HP_RES = 8 * HP_UNIT;             // units in streaming order hi0, lo0, hi1, lo1, ...; then the resident part
constexpr int RES_W1H = 0;                      // [32 row-groups][2 k-chunks][8 rows][16 B] (no swizzle), as IMG_W1
constexpr int RES_W1L = 8192;
constexpr int RES_BIAS = 16384;                 // k = 0: b1 hi, 1: b2 hi, 2: b1 lo, 3: b2 lo
constexpr int RES_W3H = 24576;                  // 4 slabs of [16 rows hi | 16 rows lo] x 128 B (SWIZZLE_128B): one N = 32 B operand
constexpr int RES_W3L = RES_W3H + 2048;         // (slab s: hi at RES_W3H + 4096 s, lo 2048 B behind it)
constexpr int RES_W3_SLAB = 4096;
constexpr int RES_B3 = 40960;                   // float [4]
constexpr int RES_ONES1 = 41216;                // every row = e0 + e2
constexpr int RES_ONES2 = 41472;                // every row = e1 + e3
constexpr int RES_BYTES = 41728;
constexpr int HP_BYTES = HP_RES + RES_BYTES;

__device__ __forceinline__ void split_f16(float v, __half& hi, __half& lo) {
    hi = __float2half_rn(v);
    lo = __float2half_rn(v - __half2float(hi));
}

__global__ void __launch_bounds__(256) hp_prepare_kernel(const float* __restrict__ W1, const float* __restrict__ b1,
                                                          const float* __restrict__ W2, const float* __restrict__ b2,
                                                          const float* __restrict__ W3, const float* __restrict__ b3,
                                                          int n_out, uint8_t* __restrict__ img) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nth = gridDim.x * blockDim.x;
    auto put2 = [&](size_t off_hi, size_t off_lo, float v) {
        __half hi, lo;
        split_f16(v, hi, lo);
        *reinterpret_cast<__half*>(img + off_hi) = hi;
        *reinterpret_cast<__half*>(img + off_lo) = lo;
    };
    for (int idx = tid; idx < TC_H * TC_H; idx += nth) {
        int k = idx / TC_H, n = idx - k * TC_H;
        int slab = k >> 6, kc = (k & 63) >> 3, ke = k & 7;
        size_t off = (size_t)n * 128 + (size_t)((kc ^ (n & 7)) * 16) + ke * 2;
        put2((size_t)(2 * slab) * HP_UNIT + off, (size_t)(2 * slab + 1) * HP_UNIT + off, W2[idx]);
    }
    uint8_t* res = img + HP_RES;
    for (int idx = tid; idx < TC_K1 * TC_H; idx += nth) {
        int k = idx / TC_H, n = idx - k * TC_H;
        size_t off = (size_t)(n >> 3) * 256 + (size_t)(k >> 3) * 128 + (size_t)(n & 7) * 16 + (k & 7) * 2;
        __half hi, lo;
        split_f16(W1[idx], hi, lo);
        *reinterpret_cast<__half*>(res + RES_W1H + off) = hi;
        *reinterpret_cast<__half*>(res + RES_W1L + off) = lo;
        __half bh1, bl1, bh2, bl2;
        split_f16(b1[n], bh1, bl1);
        split_f16(b2[n], bh2, bl2);
        __half bv = k == 0 ? bh1 : (k == 1 ? bh2 : (k == 2 ? bl1 : (k == 3 ? bl2 : __float2half_rn(0.0f))));
        *reinterpret_cast<__half*>(res + RES_BIAS + off) = bv;
    }
    for (int idx = tid; idx < TC_N3 * TC_H; idx += nth) {
        int j = idx / TC_H, k = idx - j * TC_H;
        int slab = k >> 6, kc = (k & 63) >> 3, ke = k & 7;
        size_t off = (size_t)slab * RES_W3_SLAB + (size_t)j * 128 + (size_t)((kc ^ (j & 7)) * 16) + ke * 2;
        __half hi, lo;
        split_f16(j < n_out ? W3[k * n_out + j] : 0.0f, hi, lo);
        *reinterpret_cast<__half*>(res + RES_W3H + off) = hi;
        *reinterpret_cast<__half*>(res + RES_W3L + off) = lo;
    }
    if (tid < 4) reinterpret_cast<float*>(res + RES_B3)[tid] = tid < n_out ? b3[tid] : 0.0f;
    for (int idx = tid; idx < 2 * 8 * 8; idx += nth) {
        int e = idx & 7, chunk = idx >> 6;
        *reinterpret_cast<__half*>(res + RES_ONES1 + idx * 2) = __float2half_rn((chunk == 0 && (e == 0 || e == 2)) ? 1.0f : 0.0f);
        *reinterpret_cast<__half*>(res + RES_ONES2 + idx * 2) = __float2half_rn((chunk == 0 && (e == 1 || e == 3)) ? 1.0f : 0.0f);
    }
}

// fp16 copy of the single-precision image layout of b2048_tc.cuh (W2 / W3 only are read): the backward kernel's B operands
__global__ void __launch_bounds__(256) bwd_prepare_kernel(const float* __restrict__ W2, const float* __restrict__ W3, int n_out,
                                                           uint8_t* __restrict__ img) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const int nth = gridDim.x * blockDim.x;
    for (int idx = tid; idx < TC_H * TC_H; idx += nth) {
        int k = idx / TC_H, n = idx - k * TC_H;
        int slab = k >> 6, kc = (k & 63) >> 3, ke = k & 7;
        *reinterpret_cast<__half*>(img + (size_t)IMG_W2 + (size_t)slab * 32768 + (size_t)n * 128 + (size_t)((kc ^ (n & 7)) * 16) + ke * 2) =
            __float2half_rn(W2[idx]);
    }
    for (int idx = tid; idx < TC_N3 * TC_H; idx += nth) {
        int j = idx / TC_H, k = idx - j * TC_H;
        int slab = k >> 6, kc = (k & 63) >> 3, ke = k & 7;
        *reinterpret_cast<__half*>(img + (size_t)IMG_W3 + (size_t)slab * 2048 + (size_t)j * 128 + (size_t)((kc ^ (j & 7)) * 16) + ke * 2) =
            __float2half_rn(j < n_out ? W3[k * n_out + j] : 0.0f);
    }
}

// ------------------------------------------------------------------------------------------------ pipeline context
// The three stages (forward, backward deltas, dW GEMMs) run either as separate launches over a chunk of samples (the
// images of the whole chunk go through HBM), or as ROLES of one persistent launch (update_pipe_kernel): every CTA of
// the grid is a forward, a backward or a dW CTA for the whole call, tiles of 128 samples travel from role to role
// through a ring of `R` tile slots that stays resident in the 126 MB L2, and per-tile flags (release / acquire at GPU
// scope) order the hand-offs.  The dW accumulators then live in TMEM for the whole call and the images never reach HBM.
struct PipeCtx {
    uint32_t* f_done;     // [n_tiles] forward outputs of tile t are in slot t % R      (NULL: stand-alone launch, slot == tile)
    uint32_t* b_done;     // [n_tiles] backward outputs of tile t are in its slot
    uint32_t* c2_done;    // [n_tiles] the dW2 role has consumed tile t
    uint32_t* c13_done;   // [n_tiles] the dW1 / dW3 role has consumed tile t
    int64_t R;            // ring slots
    volatile int* progress;   // debug (B2048_DBG_TC_CLOCKS): mapped host memory, 8 ints per CTA, else NULL
};
__device__ __forceinline__ void prog(const PipeCtx& px, int idx, int64_t v) {
    if (px.progress) px.progress[blockIdx.x * 8 + idx] = (int)v;
}
__device__ __forceinline__ void flag_wait(const uint32_t* p) {
    while (ld_acquire_gpu(p) == 0u) __nanosleep(100);
}
// everything this thread (and, through the mbarriers it waited on, this CTA) wrote before becomes visible to a thread that
// acquires the flag; bulk-copy (async proxy) writes must have completed (cp.async.bulk.wait_group 0) before the call
__device__ __forceinline__ void flag_set(uint32_t* p) {
    fence_proxy_async();
    __threadfence();
    st_release_gpu(p, 1u);
}

// ------------------------------------------------------------------------------------------------ precise forward
constexpr int FS_W = 0;                               // W ring: 3 slots x 32 KB
constexpr int FS_A = 3 * HP_UNIT;                     // A ring: 2 stages x [16 KB hi slab | 16 KB lo slab]
constexpr int FS_ASTAGE = 32768;
constexpr int FS_RES = FS_A + 2 * FS_ASTAGE;          // resident part of the image
constexpr int FS_A1 = FS_RES + RES_BYTES;             // [16 row-groups][2][8][16 B] = 4096 B
constexpr int FS_BAR = FS_A1 + 4096;
constexpr int FS_TOTAL = FS_BAR + 512;
static_assert(FS_RES % 1024 == 0 && (FS_RES + RES_W3H) % 1024 == 0 && (FS_RES + RES_W3L) % 1024 == 0 && FS_A1 % 128 == 0,
              "operand alignment");
static_assert(FS_TOTAL <= 232448, "fwd_hp_kernel exceeds the shared memory of an sm_100 CTA");

constexpr uint32_t kIdescF16 = idesc_f16(TC_M, TC_H);
constexpr uint32_t kIdescHeadF16 = idesc_f16(TC_M, TC_N3);
constexpr uint32_t kIdescHead32F16 = idesc_f16(TC_M, 2 * TC_N3);   // N = 32: [W3 hi | W3 lo]

struct FwdHpArgs {
    const uint8_t* img;       // split-weight image (global)
    const uint64_t* board;
    float* out;               // [n][n_out] head outputs, bias included
    uint8_t *h1, *h2;         // nullable: fp16 activation images (layout of b2048_learn_tc.cuh)
    uint64_t *m1, *m2;        // nullable: ReLU masks, entry (tile * 4 + g) * 128 + row = 64 bits of thread (row, g)
    int64_t n;
    int n_out, obs_mode;
    float obs_scale;
    long long* debug_clock;   // optional phase timestamps of CTA 0 (B2048_DBG_TC_CLOCKS), else NULL
};

constexpr int FH_THREADS = 512 + 3 * 32 + 128;   // 16 epilogue warps, MMA warp, weight loader, image storer, 4 I/O warps

// hi = fp16x2(relu(a), relu(b)) in one instruction; lo = fp16x2(relu(x) - float(hi))
__device__ __forceinline__ void relu_split(uint32_t a_bits, uint32_t b_bits, uint32_t& hi, uint32_t& lo) {
    hi = relu_pack_f16(a_bits, b_bits);
    const float2 hf = __half22float2(*reinterpret_cast<__half2*>(&hi));
    const float ra = fmaxf(__uint_as_float(a_bits), 0.0f), rb = fmaxf(__uint_as_float(b_bits), 0.0f);
    lo = pack_f16(ra - hf.x, rb - hf.y);
}

__device__ __forceinline__ void fwd_role(const FwdHpArgs& args, const PipeCtx& px, const int rank, const int nranks, uint8_t* smem) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool piped = px.f_done != nullptr;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + FS_BAR);
    const uint32_t bar_res = s_u32(&bars[0]), bar_a1 = s_u32(&bars[1]), bar_d1 = s_u32(&bars[2]), bar_d2 = s_u32(&bars[3]),
                   bar_d3 = s_u32(&bars[4]), bar_d3r = s_u32(&bars[5]), bar_out = s_u32(&bars[16]), bar_slot = s_u32(&bars[17]);
    const uint32_t w_full0 = s_u32(&bars[6]), w_empty0 = s_u32(&bars[9]);
    const uint32_t a_full0 = s_u32(&bars[12]), a_free0 = s_u32(&bars[14]);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + FS_BAR + 256);

    if (tid == 0) {
        mbar_init(bar_res, 1);
        mbar_init(bar_a1, 4);
        mbar_init(bar_d1, 1);
        mbar_init(bar_d2, 1);
        mbar_init(bar_d3, 1);
        mbar_init(bar_d3r, 4);
        mbar_init(bar_slot, 4);          // pipeline mode: the tile's ring slot is free (its previous tile has been consumed)
        mbar_init(bar_out, 20);          // pipeline mode: every epilogue / I/O warp has written its global outputs of the tile
        for (int i = 0; i < 3; ++i) { mbar_init(w_full0 + 8u * i, 1); mbar_init(w_empty0 + 8u * i, 1); }
        for (int i = 0; i < 2; ++i) { mbar_init(a_full0 + 8u * i, 16); mbar_init(a_free0 + 8u * i, 2); }
        mbar_init_fence();
    }
    // The TMEM prologue and epilogue and the two image-load loops of this role stay written out: through tmem_setup(),
    // tmem_teardown() or bulk_load_chunked() the MMA warp's loop compiles to different (equivalent) SASS.
    if (warp == 16) tmem_alloc(s_u32(tmem_slot), 512u);   // D1 = columns 0..255, D2 = 256..511, D3 = 256..271 (over D2)
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    const int64_t n_tiles = (args.n + TC_M - 1) / TC_M;
    const int64_t first = rank;

    if (warp == 16) {
        // ============================ MMA warp ============================
        // All 32 lanes walk the loops convergently (counters and descriptor words in uniform registers); lane 0 issues the
        // asynchronous instructions.  Under `if (lane == 0)` every tcgen05.mma cost ~25 vector instructions (64-bit descriptor
        // arithmetic, ELECT / R2UR per operand) and the ~100 MMAs of a tile made the warp's scalar instruction stream — not
        // shared memory — the bound of the forward role (measured the same way in b2048_mlp_gen.cu).
        {
            const bool leader = lane == 0;
            const uint8_t* gres = args.img + HP_RES;
            if (leader) {
                mbar_expect_tx(bar_res, (uint32_t)RES_BYTES);
                for (uint32_t off = 0; off < (uint32_t)RES_BYTES; off += 16384u) {
                    uint32_t sz = (uint32_t)RES_BYTES - off < 16384u ? (uint32_t)RES_BYTES - off : 16384u;
                    bulk_load(s_u32(smem + FS_RES + off), gres + off, sz, bar_res);
                }
            }
            mbar_wait(bar_res, 0);
            const uint32_t sA1 = s_u32(smem + FS_A1), sW = s_u32(smem + FS_W), sA = s_u32(smem + FS_A);
            const uint32_t sRes = s_u32(smem + FS_RES);
            const uint32_t lBias = dlo_ns(sRes + RES_BIAS), lOnes1 = dlo_ns(sRes + RES_ONES1), lOnes2 = dlo_ns(sRes + RES_ONES2);
            const uint32_t lA1 = dlo_ns(sA1), lW1H = dlo_ns(sRes + RES_W1H), lW1L = dlo_ns(sRes + RES_W1L);
            auto issue_layer1 = [&](uint32_t ph) {
                mbar_wait(bar_a1, ph);
                tc_fence_after();
                if (leader) {
                    umma_w(tmem_base, lA1, DH_NOSW, lW1H, DH_NOSW, kIdescF16, 0u);
                    umma_w(tmem_base, lA1, DH_NOSW, lW1L, DH_NOSW, kIdescF16, 1u);
                    umma_w(tmem_base, lOnes1, DH_ONES, lBias, DH_NOSW, kIdescF16, 1u);
                    umma_commit(bar_d1);
                }
            };
            uint32_t ph = 0, U = 0, F = 0;     // tile parity, streamed weight units consumed, activation ring fills consumed
            if (first < n_tiles) issue_layer1(0u);
            const bool dbg = args.debug_clock != nullptr && rank == 0 && leader;
            long long wa = 0, ww = 0, t_prev = dbg ? clock64() : 0;
            int lt = 0;
            for (int64_t tile = first; tile < n_tiles; tile += nranks, ++lt) {
                if (dbg && lt < 6) {
                    const long long now = clock64();
                    args.debug_clock[40 + 4 * lt] = now - t_prev; args.debug_clock[41 + 4 * lt] = wa; args.debug_clock[42 + 4 * lt] = ww;
                    t_prev = now; wa = 0; ww = 0;
                }
                if (tile != first) mbar_wait(bar_d3r, ph ^ 1u);     // the previous tile's head outputs have left D3 (inside D2)
                // ---- layer 2: per 64-wide K slab  D2 += H1hi W2hi + H1lo W2hi + H1hi W2lo
                for (int s = 0; s < 4; ++s) {
                    const uint32_t st = F & 1u, au = F >> 1;
                    long long c0 = dbg ? clock64() : 0;
                    mbar_wait(a_full0 + 8u * st, au & 1u);
                    tc_fence_after();
                    const uint32_t ahi = dlo_sw(sA + st * FS_ASTAGE), alo = ahi + (16384u >> 4);
                    uint32_t slot = U % 3u, use = U / 3u;
                    long long c1 = dbg ? clock64() : 0;
                    mbar_wait(w_full0 + 8u * slot, use & 1u);
                    if (dbg) { const long long c2 = clock64(); wa += c1 - c0; ww += c2 - c1; }
                    uint32_t wb = dlo_sw(sW + slot * HP_UNIT);
                    if (leader) {
                        umma_w(tmem_base + 256u, ahi, DH_SW, wb, DH_SW, kIdescF16, s ? 1u : 0u);
                        umma_w(tmem_base + 256u, ahi + 2u, DH_SW, wb + 2u, DH_SW, kIdescF16, 1u);
                        umma_w(tmem_base + 256u, ahi + 4u, DH_SW, wb + 4u, DH_SW, kIdescF16, 1u);
                        umma_w(tmem_base + 256u, ahi + 6u, DH_SW, wb + 6u, DH_SW, kIdescF16, 1u);
                        umma_w(tmem_base + 256u, alo, DH_SW, wb, DH_SW, kIdescF16, 1u);
                        umma_w(tmem_base + 256u, alo + 2u, DH_SW, wb + 2u, DH_SW, kIdescF16, 1u);
                        umma_w(tmem_base + 256u, alo + 4u, DH_SW, wb + 4u, DH_SW, kIdescF16, 1u);
                        umma_w(tmem_base + 256u, alo + 6u, DH_SW, wb + 6u, DH_SW, kIdescF16, 1u);
                        umma_commit(w_empty0 + 8u * slot);
                    }
                    ++U;
                    slot = U % 3u; use = U / 3u;
                    mbar_wait(w_full0 + 8u * slot, use & 1u);
                    wb = dlo_sw(sW + slot * HP_UNIT);
                    if (leader) {
                        umma_w(tmem_base + 256u, ahi, DH_SW, wb, DH_SW, kIdescF16, 1u);
                        umma_w(tmem_base + 256u, ahi + 2u, DH_SW, wb + 2u, DH_SW, kIdescF16, 1u);
                        umma_w(tmem_base + 256u, ahi + 4u, DH_SW, wb + 4u, DH_SW, kIdescF16, 1u);
                        umma_w(tmem_base + 256u, ahi + 6u, DH_SW, wb + 6u, DH_SW, kIdescF16, 1u);
                        umma_commit(w_empty0 + 8u * slot);
                        umma_commit(a_free0 + 8u * st);
                    }
                    ++U;
                    ++F;
                }
                if (leader) {
                    umma_w(tmem_base + 256u, lOnes2, DH_ONES, lBias, DH_NOSW, kIdescF16, 1u);
                    umma_commit(bar_d2);
                }
                // ---- the next tile's layer 1 (D1 was drained before the last H1 slab arrival waited for above)
                if (tile + nranks < n_tiles) issue_layer1(ph ^ 1u);
                // ---- head: D3 (columns 256..287: that part of D2 is drained before the first H2 slab arrives)
                for (int s = 0; s < 4; ++s) {
                    const uint32_t st = F & 1u, au = F >> 1;
                    mbar_wait(a_full0 + 8u * st, au & 1u);
                    tc_fence_after();
                    const uint32_t ahi = dlo_sw(sA + st * FS_ASTAGE), alo = ahi + (16384u >> 4);
                    // An M128 N16 K16 MMA occupies the tensor pipe as long as a full-width one (~110-140 cycles, measured in
                    // b2048_policy_tc.cu), so the three products are issued as TWO instructions per K step: H2hi x [W3hi | W3lo]
                    // as one N = 32 MMA (columns 0..15: hi x hi, 16..31: hi x lo; the reader adds the halves) and H2lo x W3hi.
                    const uint32_t w3 = dlo_sw(sRes + RES_W3H + (uint32_t)s * (uint32_t)RES_W3_SLAB);
                    if (leader) {
#pragma unroll
                        for (uint32_t q = 0; q < 4; ++q)
                            umma_w(tmem_base + 256u, ahi + 2u * q, DH_SW, w3 + 2u * q, DH_SW, kIdescHead32F16, (s | q) ? 1u : 0u);
#pragma unroll
                        for (uint32_t q = 0; q < 4; ++q) umma_w(tmem_base + 256u, alo + 2u * q, DH_SW, w3 + 2u * q, DH_SW, kIdescHeadF16, 1u);
                        umma_commit(a_free0 + 8u * st);
                    }
                    ++F;
                }
                if (leader) umma_commit(bar_d3);
                ph ^= 1u;
            }
        }
        __syncwarp();
    } else if (warp == 17) {
        // ============================ weight loader: streams the 8 split-W2 units of every tile through the ring
        if (lane == 0) {
            uint32_t U = 0;
            for (int64_t tile = first; tile < n_tiles; tile += nranks) {
                for (int j = 0; j < 8; ++j, ++U) {
                    const uint32_t slot = U % 3u, use = U / 3u;
                    if (use > 0) mbar_wait(w_empty0 + 8u * slot, (use - 1u) & 1u);
                    const uint32_t bar = w_full0 + 8u * slot;
                    mbar_expect_tx(bar, (uint32_t)HP_UNIT);
                    const uint8_t* g = args.img + (size_t)j * HP_UNIT;
                    const uint32_t d = s_u32(smem + FS_W) + slot * HP_UNIT;
#pragma unroll
                    for (uint32_t off = 0; off < (uint32_t)HP_UNIT; off += 16384u)
                        bulk_load(d + off, g + off, 16384u, bar);
                }
            }
        }
        __syncwarp();
    } else if (warp == 18) {
        // ============================ image storer: the hi half of every activation slab leaves as a global image
        if (lane == 0) {
            uint32_t F = 0;
            for (int64_t tile = first; tile < n_tiles; tile += nranks) {
                if (piped) mbar_wait(bar_slot, (uint32_t)((tile - first) / nranks) & 1u);
                for (int layer = 0; layer < 2; ++layer) {
                    uint8_t* img = layer == 0 ? args.h1 : args.h2;
                    for (int s = 0; s < 4; ++s, ++F) {
                        const uint32_t st = F & 1u, au = F >> 1;
                        mbar_wait(a_full0 + 8u * st, au & 1u);
                        if (img != nullptr) {
                            const uint32_t src = s_u32(smem + FS_A) + st * FS_ASTAGE;
#pragma unroll
                            for (int half = 0; half < 2; ++half) {
                                uint8_t* dst = img + (size_t)((tile % px.R) * 2 + half) * ACT_TILE_BYTES + (size_t)s * ACT_SLAB_BYTES;
                                bulk_store(dst, src + (uint32_t)half * 8192u, (uint32_t)ACT_SLAB_BYTES);
                            }
                            bulk_commit();
                            bulk_wait_read();
                        }
                        mbar_arrive(a_free0 + 8u * st);
                    }
                }
                if (piped) {    // publish the tile: masks / head outputs / A1^T written (bar_out), image writes complete
                    prog(px, 4, tile);
                    mbar_wait(bar_out, (uint32_t)((tile - first) / nranks) & 1u);
                    bulk_wait();
                    flag_set(px.f_done + tile);
                    prog(px, 5, tile);
                }
            }
            bulk_wait();
        }
        __syncwarp();
    } else if (warp < 16) {
        // ============================ epilogue warps ============================
        const int q = warp & 3, g = warp >> 2;
        const int row = q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t ph = 0, F = 0;
        auto epilogue = [&](uint32_t tcol0) -> uint64_t {
            uint32_t mw[4];
            uint32_t r[2][16];
            tmem_ld16_issue(tcol0 + (uint32_t)(g * 16), r[0]);      // the TMEM load of slab s + 1 is in flight while slab s is converted
#pragma unroll
            for (int s = 0; s < 4; ++s, ++F) {
                const uint32_t st = F & 1u, au = F >> 1;
                uint32_t (&rc)[16] = r[s & 1];
                tmem_ld_wait(rc);
                if (s < 3) tmem_ld16_issue(tcol0 + (uint32_t)((s + 1) * 64 + g * 16), r[(s + 1) & 1]);
                uint32_t m = 0;
#pragma unroll
                for (int i = 0; i < 16; ++i) m = __funnelshift_l(0u - rc[i], m, 1);   // z > 0  <=>  sign bit of -bits(z)
                mw[s] = m;
                if (au > 0) mbar_wait(a_free0 + 8u * st, (au - 1u) & 1u);          // the ring stage has been consumed
                uint8_t* base = smem + FS_A + st * FS_ASTAGE + row * 128;
#pragma unroll
                for (int c = 0; c < 2; ++c) {
                    uint32_t hi[4], lo[4];
#pragma unroll
                    for (int k = 0; k < 4; ++k) relu_split(rc[8 * c + 2 * k], rc[8 * c + 2 * k + 1], hi[k], lo[k]);
                    const int sw = ((g * 2 + c) ^ (row & 7)) << 4;
                    *reinterpret_cast<uint4*>(base + sw) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                    *reinterpret_cast<uint4*>(base + 16384 + sw) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                }
                fence_proxy_async_smem();
                tc_fence_before();
                __syncwarp();
                if (lane == 0) mbar_arrive(a_full0 + 8u * st);
            }
            return (uint64_t)(mw[0] | (mw[1] << 16)) | ((uint64_t)(mw[2] | (mw[3] << 16)) << 32);
        };
        int lt = 0;
        for (int64_t tile = first; tile < n_tiles; tile += nranks, ++lt) {
            const bool dbg = args.debug_clock != nullptr && rank == 0 && tid == 0 && lt < 6;
            long long* dc = dbg ? args.debug_clock + 6 * lt : nullptr;
            if (dbg) dc[0] = clock64();
            mbar_wait(bar_d1, ph);
            if (dbg) dc[1] = clock64();
            tc_fence_after();
            const uint64_t m1 = epilogue(tlane);
            if (dbg) dc[2] = clock64();
            if (piped) mbar_wait(bar_slot, ph);
            if (args.m1) args.m1[(size_t)((tile % px.R) * 4 + g) * TC_M + row] = m1;
            mbar_wait(bar_d2, ph);
            if (dbg) dc[3] = clock64();
            tc_fence_after();
            const uint64_t m2 = epilogue(tlane + 256u);
            if (dbg) dc[4] = clock64();
            if (args.m2) args.m2[(size_t)((tile % px.R) * 4 + g) * TC_M + row] = m2;
            if (piped) {
                __threadfence();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_out);
            }
            ph ^= 1u;
        }
    } else if (warp < 23) {
        // ============================ I/O warps (19..22), one thread per sample ============================
        const int q = warp & 3;   // warps 19, 20, 21, 22 -> lane quarters 3, 0, 1, 2: a TMEM load may only touch the quarter warp % 4
        const int row = q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        const float* sB3 = reinterpret_cast<const float*>(smem + FS_RES + RES_B3);
        uint32_t ph = 0;
        uint32_t pk_next[8];
        long long wait_cycles = 0;
        auto encode_a1 = [&](int64_t tile) {
            const int64_t s = tile * TC_M + row;
            uint64_t bd = (s < args.n) ? args.board[s] : 0ull;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                uint32_t e0 = (uint32_t)(bd >> (8 * j)) & 0xFu, e1 = (uint32_t)(bd >> (8 * j + 4)) & 0xFu;
                float v0, v1;
                if (args.obs_mode == B2048_OBS_RAW) { v0 = e0 ? (float)(1u << e0) : 0.0f; v1 = e1 ? (float)(1u << e1) : 0.0f; }
                else { v0 = (float)e0 * args.obs_scale; v1 = (float)e1 * args.obs_scale; }
                pk_next[j] = pack_f16(v0, v1);
            }
            uint8_t* a1 = smem + FS_A1 + (row >> 3) * 256 + (row & 7) * 16;
            *reinterpret_cast<uint4*>(a1) = make_uint4(pk_next[0], pk_next[1], pk_next[2], pk_next[3]);
            *reinterpret_cast<uint4*>(a1 + 128) = make_uint4(pk_next[4], pk_next[5], pk_next[6], pk_next[7]);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_a1);
        };
        if (first < n_tiles) encode_a1(first);
        mbar_wait(bar_res, 0);
        for (int64_t tile = first; tile < n_tiles; tile += nranks) {
            const int64_t s = tile * TC_M + row;
            const int64_t srow = (tile % px.R) * TC_M + row;                      // row inside the ring of tile slots
            mbar_wait(bar_d1, ph);                                               // A1 is free
            if (piped) {
                // The tile's slot is taken only now (not when its inputs were prefetched): its previous tile has been
                // consumed by both dW roles (hence by the backward role).  The storer and the epilogue warps write
                // into the slot after bar_slot.
                if (tile >= px.R && lane == 0) {
                    const long long w0 = clock64();
                    flag_wait(px.c2_done + (tile - px.R));
                    flag_wait(px.c13_done + (tile - px.R));
                    if (warp == 19) { wait_cycles += clock64() - w0; prog(px, 6, wait_cycles >> 10); }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_slot);
            }
            const int64_t next = tile + nranks;
            if (next < n_tiles) encode_a1(next);
            mbar_wait(bar_d3, ph);
            tc_fence_after();
            uint32_t r4[4], r4b[4];
            tmem_ld4_issue(tlane + 256u, r4);
            tmem_ld4_issue(tlane + 256u + 16u, r4b);            // the hi x lo partial sums
            tmem_ld_wait(r4);                                   // covers both loads
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_d3r);
            if (s < args.n) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < args.n_out) args.out[srow * args.n_out + j] = (__uint_as_float(r4[j]) + __uint_as_float(r4b[j])) + sB3[j];
            }
            if (piped) {
                __threadfence();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_out);
            }
            ph ^= 1u;
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 16) tmem_dealloc(tmem_base, 512u);
}

__global__ void __launch_bounds__(FH_THREADS, 1) fwd_hp_kernel(const __grid_constant__ FwdHpArgs args) {
    extern __shared__ __align__(1024) uint8_t smem[];
    PipeCtx px;
    px.f_done = nullptr; px.b_done = nullptr; px.c2_done = nullptr; px.c13_done = nullptr;
    px.R = (args.n + TC_M - 1) / TC_M + 1;      // stand-alone: slot == tile
    fwd_role(args, px, (int)blockIdx.x, (int)gridDim.x, smem);
}

// ------------------------------------------------------------------------------------------------ backward deltas
constexpr int BW_D3A = SM_BAR + 256;     // head deltas of the tile in flight as an fp16 A operand [128 x 16], A1's layout
constexpr int BW_TOTAL = BW_D3A + 4096;
constexpr int BW_A1T = IMG_W1;           // 2 buffers x 2 half-tiles x [32 rows x 128 B]: inputs^T (+ a ones row) of the tile, K-major
                                         // B operand of dW1^T = DL1^T A1; lives in the W1 / BIAS part of the image area (not loaded)
static_assert(BW_TOTAL <= 232448, "bwd_tc_kernel exceeds the shared memory of an sm_100 CTA");
static_assert(IMG_W3 - IMG_W1 >= 2 * 8192 && BW_A1T % 1024 == 0, "A1^T buffers");

struct BwdArgs {
    const uint8_t* img;           // fp16 image, layout of b2048_tc.cuh (W2 and W3 are read)
    const float* logits;          // [n][n_out] from fwd_hp_kernel (head_mode 0)
    const uint64_t *m1, *m2;      // ReLU masks from fwd_hp_kernel
    const uint64_t* board;        // packed boards (inputs of dW1)
    const uint8_t* mask_flags;
    const uint8_t* action;
    const float* coef;
    const float* scale;           // device float[2]: loss scale S (a power of two) and 1 / S
    uint8_t *dl2, *d3t;
    float *gW1, *gb1, *gb3;
    int64_t n;
    int head_mode, n_out, obs_mode;
    float obs_scale;
    long long* debug_clock;   // optional phase timestamps of CTA 0 (B2048_DBG_TC_CLOCKS), else NULL
};

// The entropy variant's extra arguments: per-sample ecoef and the optional sum of H over the valid samples.
struct BwdEnt {
    const float* ent_coef;
    double* ent_sum;              // nullable
};
struct BwdEntArgs {
    BwdArgs b;
    BwdEnt e;
};

constexpr int BW_THREADS = 512 + 32 + 128;

// Backward deltas of one 128-sample tile at a time, and the input-layer gradient:
//   D5 = d3 W3^T in two N = 128 halves (TMEM columns 0..127, the second half once the first is drained)
//   DL2 = D5 . [z2 > 0]  -> A2 (fp16, the A operand of D4) and the global DL2 image (dW2 is another kernel / role)
//   D4 = DL2 W2 (TMEM columns 256..511)  ->  DL1 = D4 . [z1 > 0]  -> A2
//   dW1^T += DL1^T [A1 | 1]  (TMEM columns 128..191, N = 32: columns 0..15 = the 16 inputs, column 16 = the bias gradient);
//   DL1 never leaves the SM; the accumulators stay in TMEM for all tiles of the CTA and are added to the gradient once.
// kEnt: the policy head's delta carries the entropy bonus, d_j = coef (1[a = j] - p_j) - ecoef t_j (b2048_entropy.cuh)
template <bool kEnt>
__device__ __forceinline__ void bwd_role(const BwdArgs& args, const BwdEnt& ent, const PipeCtx& px, const int rank, const int nranks,
                                         uint8_t* smem) {
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const bool piped = px.f_done != nullptr;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + SM_BAR);
    const uint32_t bar_img = s_u32(&bars[0]), bar_dl3 = s_u32(&bars[1]), bar_d5 = s_u32(&bars[2]), bar_d4 = s_u32(&bars[3]),
                   bar_free = s_u32(&bars[4]), bar_d5b = s_u32(&bars[5]);
    const uint32_t bar_bslab0 = s_u32(&bars[8]);    // [8..11]  DL2 slab written (D5 drained for that slab)
    const uint32_t bar_dslab0 = s_u32(&bars[12]);   // [12..15] DL1 slab written (D4 drained for that slab)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + SM_BAR + 208);

    if (tid == 0) {
        mbar_init(bar_img, 1);
        mbar_init(bar_dl3, 4);
        mbar_init(bar_d5, 1);
        mbar_init(bar_d5b, 1);
        mbar_init(bar_d4, 1);
        mbar_init(bar_free, 1);          // the dW1 MMAs of the tile have completed: A2 and the tile's A1^T buffer are free
        for (int g = 0; g < 4; ++g) {
            mbar_init(bar_bslab0 + 8u * g, 16);
            mbar_init(bar_dslab0 + 8u * g, 16);
        }
        mbar_init_fence();
    }
    const uint32_t tmem_base = tmem_setup(warp == 16, tmem_slot, 512u);
    const int64_t n_tiles = (args.n + TC_M - 1) / TC_M;
    const int64_t first = rank;
    const int64_t n_local = first < n_tiles ? (n_tiles - first + nranks - 1) / nranks : 0;

    if (warp == 16) {
        // ============================ MMA / copy warp ============================
        if (lane == 0) {
            const uint32_t sA2 = s_u32(smem + SM_A2), sW2 = s_u32(smem + IMG_W2), sW3 = s_u32(smem + IMG_W3);
            const uint32_t sA1T = s_u32(smem + BW_A1T);
            constexpr uint32_t kIdescBwd = kIdescF16 | kIdescBMn;                                                          // M128 N256
            constexpr uint32_t kIdescD5 = idesc_f16(128, 128) | kIdescBMn;
            constexpr uint32_t kIdescDw1 = idesc_f16(128, 32) | kIdescAMn;
            // only W2 and W3 of the image are read by this kernel
            mbar_expect_tx(bar_img, (uint32_t)(131072 + 8192));
            bulk_load_chunked<16384u>(s_u32(smem + IMG_W2), args.img + IMG_W2, 131072u, bar_img);
            bulk_load(s_u32(smem + IMG_W3), args.img + IMG_W3, 8192u, bar_img);
            mbar_wait(bar_img, 0);
            auto issue_d5a = [&](uint32_t ph) {
                // backward through the head, features 0..127: D5 = d3 . W3^T.  A = d3 as fp16 [128 x 16] (K-major, A1's layout);
                // B = the head's W3 image [j][f] read MN-major (N = f contiguous: 64-wide slabs 2048 B apart, 8 K rows = 1024 B)
                mbar_wait(bar_dl3, ph);
                tc_fence_after();
                umma_f16(tmem_base, desc_nosw_k16(s_u32(smem + BW_D3A)), desc_sw128_mn(sW3, 2048u), kIdescD5, 0u);
                umma_commit(bar_d5);
            };
            uint32_t ph = 0;
            int64_t lt = 0;
            if (first < n_tiles) issue_d5a(0u);
            for (int64_t tile = first; tile < n_tiles; tile += nranks, ++lt) {
                // ---- backward through layer 2: D4 = DL2 . W2 over K = out features; B = the W2 image [out][in] read
                //      MN-major (N = in contiguous: 64-wide slabs 32768 B apart, 8 K rows = 1024 B)
                for (int g = 0; g < 4; ++g) {
                    mbar_wait(bar_bslab0 + 8u * g, ph);
                    tc_fence_after();
                    if (g == 1) {   // slabs 0 and 1 of DL2 are written, i.e. the first half of D5 is drained: features 128..255
                        umma_f16(tmem_base, desc_nosw_k16(s_u32(smem + BW_D3A)), desc_sw128_mn(sW3 + 2u * 2048u, 2048u), kIdescD5, 0u);
                        umma_commit(bar_d5b);
                    }
#pragma unroll
                    for (int q = 0; q < 4; ++q)
                        umma_f16(tmem_base + 256u, desc_sw128(sA2 + (uint32_t)g * 16384u + (uint32_t)q * 32u),
                                 desc_sw128_mn(sW2 + (uint32_t)(g * 64 + q * 16) * 128u, 32768u), kIdescBwd, (g | q) ? 1u : 0u);
                    store_act_slab(args.dl2, tile % px.R, sA2, g);
                }
                bulk_commit();
                bulk_wait_read();                        // epilogue 4 overwrites DL2 once bar_d4 completes
                umma_commit(bar_d4);
                // ---- the next tile's D5 (this tile's D5 was drained by every warp before the DL2 slab arrivals)
                if (tile + nranks < n_tiles) issue_d5a(ph ^ 1u);
                // ---- dW1^T += DL1^T [A1 | 1]: A = DL1 in A2 read MN-major (M = features: 64-wide slabs 16384 B apart,
                //      K = samples: 8 rows = 1024 B), B = the tile's A1^T buffer (K-major, 32 rows: 16 inputs, the ones row, zeros)
                for (int g = 0; g < 4; ++g) mbar_wait(bar_dslab0 + 8u * g, ph);
                tc_fence_after();
                const uint32_t sB = sA1T + (uint32_t)(lt & 1) * 8192u;
#pragma unroll
                for (int kk = 0; kk < 8; ++kk) {         // 16 samples per MMA
                    const uint64_t db = desc_sw128(sB + (uint32_t)(kk >> 2) * 4096u + (uint32_t)(kk & 3) * 32u);
#pragma unroll
                    for (int hf = 0; hf < 2; ++hf)
                        umma_f16(tmem_base + 128u + (uint32_t)(hf * 32), desc_sw128_mn(sA2 + (uint32_t)hf * 32768u + (uint32_t)kk * 2048u, 16384u),
                                 db, kIdescDw1, (lt | kk) ? 1u : 0u);
                }
                umma_commit(bar_free);
                if (piped) {                             // publish the tile: d3^T written, DL2 image writes complete
                    prog(px, 4, tile);
                    bulk_wait();
                    flag_set(px.b_done + tile);
                    prog(px, 5, tile);
                }
                ph ^= 1u;
            }
            bulk_wait();
        }
        __syncwarp();
    } else if (warp < 16) {
        // ============================ epilogue warps ============================
        const int q = warp & 3, g = warp >> 2;
        const int row = q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        uint8_t* a2_row = smem + SM_A2 + row * 128;
        uint32_t ph = 0;
        // slab s of the [128 x 256] delta tile: columns tcol .. tcol + 15 of this warp's lanes, masked, as fp16 into A2
        auto masked_slab = [&](uint32_t tcol, int s, uint64_t mask, uint32_t bar0) {
            uint32_t rr[16];
            tmem_ld16(tcol, rr);
            const uint32_t mb = (uint32_t)(mask >> (16 * s)) & 0xFFFFu;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                uint32_t out[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int i0 = c * 8 + 2 * k;
                    float lo = (mb >> (15 - i0)) & 1u ? __uint_as_float(rr[i0]) : 0.0f;
                    float hi = (mb >> (14 - i0)) & 1u ? __uint_as_float(rr[i0 + 1]) : 0.0f;
                    out[k] = pack_f16(lo, hi);
                }
                const int sw = ((g * 2 + c) ^ (row & 7)) << 4;
                *reinterpret_cast<uint4*>(a2_row + s * 16384 + sw) = make_uint4(out[0], out[1], out[2], out[3]);
            }
            fence_proxy_async_smem();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar0 + 8u * s);
        };
        int lt = 0;
        long long wait_cycles = 0;
        for (int64_t tile = first; tile < n_tiles; tile += nranks, ++lt) {
            const bool dbg = args.debug_clock != nullptr && rank == 0 && tid == 0 && lt < 6;
            long long* dc = dbg ? args.debug_clock + 8 * lt : nullptr;
            if (dbg) dc[0] = clock64();
            if (piped) {
                if (lane == 0) {
                    const long long w0 = clock64();
                    flag_wait(px.f_done + tile);
                    if (warp == 0) { wait_cycles += clock64() - w0; prog(px, 6, wait_cycles >> 10); }
                }
                __syncwarp();
            }
            const uint64_t m2 = args.m2[(size_t)((tile % px.R) * 4 + g) * TC_M + row];
            const uint64_t m1 = args.m1[(size_t)((tile % px.R) * 4 + g) * TC_M + row];
            // ---- DL2 = D5 [z2 > 0]  (A2 is free once the previous tile's dW1 MMAs have read DL1)
            mbar_wait(bar_d5, ph);
            if (dbg) dc[1] = clock64();
            if (tile != first) mbar_wait(bar_free, ph ^ 1u);
            if (dbg) dc[2] = clock64();
            tc_fence_after();
            masked_slab(tlane + (uint32_t)(g * 16), 0, m2, bar_bslab0);
            masked_slab(tlane + (uint32_t)(64 + g * 16), 1, m2, bar_bslab0);
            mbar_wait(bar_d5b, ph);                      // features 128..255 of D5 (same TMEM columns)
            tc_fence_after();
            masked_slab(tlane + (uint32_t)(g * 16), 2, m2, bar_bslab0);
            masked_slab(tlane + (uint32_t)(64 + g * 16), 3, m2, bar_bslab0);
            if (dbg) dc[3] = clock64();
            // ---- DL1 = D4 [z1 > 0] over DL2 (the backward MMAs have completed); read by the dW1 MMAs
            mbar_wait(bar_d4, ph);
            if (dbg) dc[4] = clock64();
            tc_fence_after();
#pragma unroll
            for (int s = 0; s < 4; ++s) masked_slab(tlane + 256u + (uint32_t)(s * 64 + g * 16), s, m1, bar_dslab0);
            if (dbg) dc[5] = clock64();
            ph ^= 1u;
        }
        // ---- read-out of dW1^T (columns 0..15) and db1 (column 16): lane quarter q, features hf * 128 + q * 32 + lane
        if (g == 0 && n_local > 0) {
            mbar_wait(bar_free, ph ^ 1u);                // the last tile's dW1 MMAs
            tc_fence_after();
            const float inv = args.scale[1];
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                const int m = hf * 128 + row;
                uint32_t r0[16], r1[16];
                tmem_ld16(tlane + 128u + (uint32_t)(hf * 32), r0);
                tmem_ld16(tlane + 128u + (uint32_t)(hf * 32 + 16), r1);
#pragma unroll
                for (int i = 0; i < 16; ++i) {
                    const float v = __uint_as_float(r0[i]) * inv;
                    if (v != 0.0f) atomicAdd(args.gW1 + (size_t)i * TC_H + m, v);          // dW1[k][m]
                }
                const float vb = __uint_as_float(r1[0]) * inv;
                if (vb != 0.0f) atomicAdd(args.gb1 + m, vb);
            }
        }
    } else if (warp < 21) {
        // ============================ I/O warps (17..20), one thread per sample ============================
        const int row = (warp & 3) * 32 + lane;
        uint8_t* d3a = smem + BW_D3A + (row >> 3) * 256 + (row & 7) * 16;   // this row's two 16-byte K chunks
        *reinterpret_cast<uint4*>(d3a + 128) = make_uint4(0u, 0u, 0u, 0u);    // k = 8..15 stay zero
        // A1^T buffers: rows 17..31 stay zero, row 16 = 1 (the bias-gradient column), rows 0..15 are rewritten per tile
        {
            const int tq = tid - 17 * 32;                                      // 0..127
            for (int i = tq; i < 2 * 8192 / 16; i += 128) {
                const int off = i * 16, rowj = (off & 4095) >> 7;
                const uint32_t v = rowj == 16 ? 0x3C003C00u : 0u;              // fp16 1.0 pairs
                *reinterpret_cast<uint4*>(smem + BW_A1T + off) = make_uint4(v, v, v, v);
            }
            bar_sync(1, 128);                     // the four I/O warps only
        }
        const float S = args.scale[0];
        uint32_t ph = 0;
        int64_t lt = 0;
        for (int64_t tile = first; tile < n_tiles; tile += nranks, ++lt) {
            const int64_t s = tile * TC_M + row;
            const int64_t srow = (tile % px.R) * TC_M + row;                      // row inside the ring of tile slots
            const bool valid = s < args.n;
            const bool use_mask = args.mask_flags != nullptr;
            uint32_t fl = 0xFu, act = 0;
            float cf = 0.0f, ecf = 0.0f, lg[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            const uint64_t bd = valid ? args.board[s] : 0ull;
            if (piped) {
                if (lane == 0) flag_wait(px.f_done + tile);
                __syncwarp();
            }
            if (valid) {
                if (use_mask) fl = args.mask_flags[s];
                if (args.action) act = args.action[s];
                cf = args.coef[s];
                if constexpr (kEnt) ecf = ent.ent_coef[s];
                if (args.head_mode == 0) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (j < args.n_out) lg[j] = args.logits[srow * args.n_out + j];
                }
            }
            float d[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            if (args.head_mode == 0) {
                float m[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) m[j] = (use_mask && !((fl >> j) & 1u)) ? -1e9f : lg[j];   // MLP.py:144-146
                const float mx = fmaxf(fmaxf(m[0], m[1]), fmaxf(m[2], m[3]));
                float e[4], sum = 0.0f;
#pragma unroll
                for (int j = 0; j < 4; ++j) { e[j] = expf(m[j] - mx); sum += e[j]; }
                if constexpr (kEnt) {
                    float z[4], p[4], t[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) { z[j] = m[j] - mx; p[j] = e[j] / sum; }
                    const float H = entropy_row(z, logf(sum), p, use_mask ? fl : 0xFu, args.n_out, t);
#pragma unroll
                    for (int j = 0; j < 4; ++j) d[j] = cf * ((act == (uint32_t)j ? 1.0f : 0.0f) - p[j]) - ecf * t[j];
                    if (ent.ent_sum) {                                            // one float64 atomic per warp and tile
                        float hs = valid ? H : 0.0f;
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) hs += __shfl_xor_sync(0xFFFFFFFFu, hs, o);
                        if (lane == 0 && hs != 0.0f) atomicAdd(ent.ent_sum, (double)hs);
                    }
                } else {
#pragma unroll
                    for (int j = 0; j < 4; ++j) d[j] = cf * ((act == (uint32_t)j ? 1.0f : 0.0f) - e[j] / sum);   // reinforce_agent.py:340-344
                }
            } else {
                d[0] = cf;                                                        // value head: dLoss/dV * weight
            }
            const uint32_t p01 = pack_f16(d[0] * S, d[1] * S), p23 = pack_f16(d[2] * S, d[3] * S);
            const uint32_t pk[2] = {p01, p23};
            // transposed fp16 copy for dW3 = H2^T d3 (rows >= n_out of the small image stay zero).  Pipeline mode: written
            // BEFORE the arrival that lets the MMA lane issue this tile's D5, so the lane's later publication of the tile
            // (which follows that wait in program order) covers it; stand-alone it stays off the critical path.
            if (piped) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < args.n_out)
                        *reinterpret_cast<uint16_t*>(args.d3t + small_off(srow, j)) = (uint16_t)(pk[j >> 1] >> (16 * (j & 1)));
                __threadfence();
            }
            // the tile's inputs, transposed, into its A1^T buffer (two tiles back used the same buffer: its dW1 MMAs are done)
            if (lt >= 2) mbar_wait(bar_free, ph);
            {
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const uint32_t e = (uint32_t)(bd >> (4 * j)) & 0xFu;
                    const float v = args.obs_mode == B2048_OBS_RAW ? (e ? (float)(1u << e) : 0.0f) : (float)e * args.obs_scale;
                    // element (row j, sample r): j * 128 + (((r >> 3) ^ (j & 7)) << 4) + (r & 7) * 2
                    uint8_t* pz = smem + BW_A1T + (lt & 1) * 8192 + (row >> 6) * 4096 + j * 128 +
                                  ((((row & 63) >> 3) ^ (j & 7)) << 4) + (row & 7) * 2;
                    *reinterpret_cast<__half*>(pz) = __float2half_rn(v);
                }
            }
            if (tile != first) mbar_wait(bar_d5b, ph ^ 1u);                       // the previous tile's D5 (both halves) has read d3a
            *reinterpret_cast<uint4*>(d3a) = make_uint4(p01, p23, 0u, 0u);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_dl3);
            if (!piped) {
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (j < args.n_out)
                        *reinterpret_cast<uint16_t*>(args.d3t + small_off(srow, j)) = (uint16_t)(pk[j >> 1] >> (16 * (j & 1)));
            }
            // the head bias gradient (unscaled float32 sum over the warp's 32 samples)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                float v = d[j];
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
                if (lane == 0 && j < args.n_out && v != 0.0f) atomicAdd(args.gb3 + j, v);
            }
            ph ^= 1u;
        }
    }

    tmem_teardown(warp == 16, tmem_base, 512u);
}

__global__ void __launch_bounds__(BW_THREADS, 1) bwd_tc_kernel(const __grid_constant__ BwdArgs args) {
    extern __shared__ __align__(1024) uint8_t smem[];
    PipeCtx px;
    px.f_done = nullptr; px.b_done = nullptr; px.c2_done = nullptr; px.c13_done = nullptr;
    px.R = (args.n + TC_M - 1) / TC_M + 1;      // stand-alone: slot == tile
    bwd_role<false>(args, BwdEnt{}, px, (int)blockIdx.x, (int)gridDim.x, smem);
}

__global__ void __launch_bounds__(BW_THREADS, 1) bwd_tc_ent_kernel(const __grid_constant__ BwdEntArgs args) {
    extern __shared__ __align__(1024) uint8_t smem[];
    PipeCtx px;
    px.f_done = nullptr; px.b_done = nullptr; px.c2_done = nullptr; px.c13_done = nullptr;
    px.R = (args.b.n + TC_M - 1) / TC_M + 1;    // stand-alone: slot == tile
    bwd_role<true>(args.b, args.e, px, (int)blockIdx.x, (int)gridDim.x, smem);
}

// ------------------------------------------------------------------------------------------------ dW roles
// The dW GEMMs of atb_tc_kernel (b2048_learn_tc.cu) as roles of the persistent pipeline: a CTA takes the tiles rank,
// rank + nranks, ... as the backward role publishes them, pulls the two 64-sample halves of the tile's images from the L2-resident
// ring with bulk copies (3-stage ring) and accumulates in TMEM for the WHOLE call — one read-out + atomic add per CTA and call.
//   kWhich == 2 : dW2 = H1^T DL2 (2 x 256 TMEM columns), db2 = column sums of DL2
//   kWhich == 3 : dW3 = H2^T d3 (2 x 16 TMEM columns)
// (dW1 and db1 are accumulated by the backward role itself: DL1 never leaves its SM.)
struct DwArgs {
    const uint8_t *h1, *h2, *dl2, *d3t;   // the ring's images
    float *gW2, *gb2, *gW3;
    const float* inv_scale;                           // device float: 1 / loss scale
    int64_t n_tiles;
    int n_out;
};
template <int kWhich>
struct DwCfg {
    static constexpr int kStageBytes = kWhich == 2 ? 2 * ACT_TILE_BYTES : ACT_TILE_BYTES + SMALL_TILE_BYTES;
    static constexpr int kStages = kWhich == 2 ? 3 : 6;
    static constexpr int kBar = kStages * kStageBytes;
    static constexpr int kSmem = kBar + 256;
    static constexpr uint32_t kTmemCols = kWhich == 2 ? 512u : 32u;
};
static_assert(DwCfg<2>::kSmem <= 232448 && DwCfg<2>::kStageBytes % 1024 == 0 && DwCfg<3>::kStageBytes % 1024 == 0, "dW role stages");

__device__ __forceinline__ float2 h2f(uint32_t w) { return __half22float2(*reinterpret_cast<const __half2*>(&w)); }

template <int kWhich>
__device__ __forceinline__ void dw_role(const DwArgs& args, const PipeCtx& px, const int rank, const int nranks, uint8_t* smem) {
    using Cfg = DwCfg<kWhich>;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + Cfg::kBar);
    const uint32_t bar_full0 = s_u32(&bars[0]), bar_empty0 = s_u32(&bars[8]), bar_done = s_u32(&bars[16]);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + Cfg::kBar + 160);
    if (tid == 0) {
        for (int i = 0; i < Cfg::kStages; ++i) {
            mbar_init(bar_full0 + 8u * i, 1);
            mbar_init(bar_empty0 + 8u * i, kWhich == 2 ? 5 : 1);   // the MMA commit (+ the four column-sum warps of the dW2 role)
        }
        mbar_init(bar_done, 1);
        mbar_init_fence();
    }
    const uint32_t tmem_base = tmem_setup(warp == 1, tmem_slot, Cfg::kTmemCols);
    const int64_t n_my = rank < args.n_tiles ? (args.n_tiles - rank + nranks - 1) / nranks : 0;
    const int64_t n_it = 2 * n_my;                          // 64-sample half tiles
    uint32_t* c_done = kWhich == 2 ? px.c2_done : px.c13_done;      // (c13_done: the dW3 role)

    if (warp == 0) {
        if (lane == 0) {
            long long wait_cycles = 0;
            for (int64_t it = 0; it < n_it; ++it) {
                const int st = (int)(it % Cfg::kStages);
                const int64_t use = it / Cfg::kStages;
                const int64_t tile = rank + (it >> 1) * nranks;
                const int64_t half = (tile % px.R) * 2 + (it & 1);
                if (use > 0) mbar_wait(bar_empty0 + 8u * st, (uint32_t)(use - 1) & 1u);
                if ((it & 1) == 0) {
                    const long long w0 = clock64();
                    flag_wait(px.b_done + tile);             // forward and backward outputs of the tile are in its slot
                    wait_cycles += clock64() - w0;
                    prog(px, 6, wait_cycles >> 10);
                    fence_proxy_async();
                }
                const uint32_t bar = bar_full0 + 8u * st;
                mbar_expect_tx(bar, (uint32_t)Cfg::kStageBytes);
                const uint32_t sa = s_u32(smem + st * Cfg::kStageBytes);
                const uint8_t* ga = (kWhich == 2 ? args.h1 : args.h2) + (size_t)half * ACT_TILE_BYTES;
                bulk_load_chunked<16384u>(sa, ga, (uint32_t)ACT_TILE_BYTES, bar);
                if (kWhich == 2) {
                    const uint8_t* gb = args.dl2 + (size_t)half * ACT_TILE_BYTES;
                    bulk_load_chunked<16384u>(sa + (uint32_t)ACT_TILE_BYTES, gb, (uint32_t)ACT_TILE_BYTES, bar);
                } else {
                    bulk_load(sa + (uint32_t)ACT_TILE_BYTES, args.d3t + (size_t)half * SMALL_TILE_BYTES, (uint32_t)SMALL_TILE_BYTES, bar);
                }
            }
        }
        __syncwarp();
    } else if (warp == 6) {
        // ---- releaser: a tile's slot is handed back as soon as the MMAs (and column sums) of its second half have completed
        if (lane == 0) {
            for (int64_t j = 0; j < n_it; ++j) {
                mbar_wait(bar_empty0 + 8u * (uint32_t)(j % Cfg::kStages), (uint32_t)(j / Cfg::kStages) & 1u);
                if (j & 1) st_release_gpu(c_done + rank + (j >> 1) * nranks, 1u);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            constexpr uint32_t idesc2 = idesc_f16(128, 256) | kIdescAMn | kIdescBMn;
            constexpr uint32_t idesc16 = idesc_f16(128, 16) | kIdescAMn;
            for (int64_t it = 0; it < n_it; ++it) {
                const int st = (int)(it % Cfg::kStages);
                const int64_t use = it / Cfg::kStages;
                mbar_wait(bar_full0 + 8u * st, (uint32_t)use & 1u);
                tc_fence_after();
                const uint32_t sa = s_u32(smem + st * Cfg::kStageBytes), sb = sa + (uint32_t)ACT_TILE_BYTES;
                const uint32_t acc = it ? 1u : 0u;
#pragma unroll
                for (int kk = 0; kk < 4; ++kk) {                                   // 16 samples per MMA
                    if (kWhich == 2) {
                        const uint64_t db = desc_sw128_mn(sb + (uint32_t)kk * 2048u, ACT_SLAB_BYTES);
#pragma unroll
                        for (int hf = 0; hf < 2; ++hf)
                            umma_f16(tmem_base + (uint32_t)(hf * 256), desc_sw128_mn(sa + (uint32_t)hf * 16384u + (uint32_t)kk * 2048u, ACT_SLAB_BYTES),
                                     db, idesc2, (acc | (uint32_t)kk) ? 1u : 0u);
                    } else {
#pragma unroll
                        for (int hf = 0; hf < 2; ++hf)
                            umma_f16(tmem_base + (uint32_t)(hf * 16), desc_sw128_mn(sa + (uint32_t)hf * 16384u + (uint32_t)kk * 2048u, ACT_SLAB_BYTES),
                                     desc_sw128(sb + (uint32_t)kk * 32u), idesc16, (acc | (uint32_t)kk) ? 1u : 0u);
                    }
                }
                umma_commit(bar_empty0 + 8u * st);
            }
            umma_commit(bar_done);
        }
        __syncwarp();
    } else if (warp < 6) {
        // ---- column sums of the staged DL image (DL2 is the second image of a dW2 stage, DL1 the second of a dW1/dW3 stage)
        const int cw = warp - 2, chunk = lane & 7, rsub = lane >> 3;
        float acc[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[e] = 0.0f;
        for (int64_t it = 0; kWhich == 2 && it < n_it; ++it) {
            const int st = (int)(it % Cfg::kStages);
            const int64_t use = it / Cfg::kStages;
            mbar_wait(bar_full0 + 8u * st, (uint32_t)use & 1u);
            const uint8_t* x = smem + st * Cfg::kStageBytes + ACT_TILE_BYTES + cw * ACT_SLAB_BYTES;
#pragma unroll 4
            for (int r = rsub; r < 64; r += 4) {
                const uint4 v = *reinterpret_cast<const uint4*>(x + r * 128 + ((chunk ^ (r & 7)) << 4));
                const float2 f0 = h2f(v.x), f1 = h2f(v.y), f2 = h2f(v.z), f3 = h2f(v.w);
                acc[0] += f0.x; acc[1] += f0.y; acc[2] += f1.x; acc[3] += f1.y; acc[4] += f2.x; acc[5] += f2.y; acc[6] += f3.x; acc[7] += f3.y;
            }
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_empty0 + 8u * st);
        }
        const float out_scale = *args.inv_scale;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            acc[e] += __shfl_xor_sync(0xFFFFFFFFu, acc[e], 8);
            acc[e] += __shfl_xor_sync(0xFFFFFFFFu, acc[e], 16);
        }
        float* gb = args.gb2;
        if (kWhich == 2 && lane < 8 && n_it > 0) {
#pragma unroll
            for (int e = 0; e < 8; ++e)
                if (acc[e] != 0.0f) atomicAdd(gb + cw * 64 + chunk * 8 + e, acc[e] * out_scale);
        }
        // ---- read-out: TMEM lane quarter = warp % 4
        if (n_it > 0) {
            mbar_wait(bar_done, 0);
            tc_fence_after();
            const int q = warp & 3;
            const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {
                const int m = hf * 128 + q * 32 + lane;                        // feature index
                if (kWhich == 2) {
                    for (int c0 = 0; c0 < 256; c0 += 16) {
                        uint32_t r[16];
                        tmem_ld16(tlane + (uint32_t)(hf * 256 + c0), r);
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const float v = __uint_as_float(r[i]) * out_scale;
                            if (v != 0.0f) atomicAdd(args.gW2 + (size_t)m * TC_H + (c0 + i), v);
                        }
                    }
                } else {
                    uint32_t r3[16];
                    tmem_ld16(tlane + (uint32_t)(hf * 16), r3);
#pragma unroll
                    for (int i = 0; i < 16; ++i) {
                        const float v3 = __uint_as_float(r3[i]) * out_scale;
                        if (i < args.n_out && v3 != 0.0f) atomicAdd(args.gW3 + (size_t)m * args.n_out + i, v3);       // dW3[m][j]
                    }
                }
            }
        }
    }
    tmem_teardown(warp == 1, tmem_base, Cfg::kTmemCols);
}

// ------------------------------------------------------------------------------------------------ the persistent update pipeline
struct PipeArgs {
    FwdHpArgs f;
    BwdArgs b;
    DwArgs d;
    PipeCtx px;
    int nF, nB, nC2, nC13;     // CTAs per role: forward, backward (+ dW1), dW2, dW3 (sum == gridDim.x)
};
constexpr int PIPE_SMEM = FS_TOTAL > BW_TOTAL ? (FS_TOTAL > DwCfg<3>::kSmem ? FS_TOTAL : DwCfg<3>::kSmem)
                                              : (BW_TOTAL > DwCfg<3>::kSmem ? BW_TOTAL : DwCfg<3>::kSmem);
static_assert(PIPE_SMEM <= 232448 && DwCfg<2>::kSmem <= PIPE_SMEM, "update_pipe_kernel shared memory");

__global__ void __launch_bounds__(FH_THREADS, 1) update_pipe_kernel(const __grid_constant__ PipeArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    int r = (int)blockIdx.x;
    const long long t0 = clock64();
    if (threadIdx.x == 0) prog(a.px, 0, r < a.nF ? 100 : (r < a.nF + a.nB ? 200 : (r < a.nF + a.nB + a.nC2 ? 300 : 400)));
    if (r < a.nF) fwd_role(a.f, a.px, r, a.nF, smem);
    else if (r < a.nF + a.nB) bwd_role<false>(a.b, BwdEnt{}, a.px, r - a.nF, a.nB, smem);
    else if (r < a.nF + a.nB + a.nC2) dw_role<2>(a.d, a.px, r - a.nF - a.nB, a.nC2, smem);
    else dw_role<3>(a.d, a.px, r - a.nF - a.nB - a.nC2, a.nC13, smem);
    if (threadIdx.x == 0) prog(a.px, 7, (clock64() - t0) >> 10);
}

// The pipeline with the entropy bonus in the backward role: same roles, role split and shared memory as update_pipe_kernel.
struct PipeEntArgs {
    FwdHpArgs f;
    BwdArgs b;
    DwArgs d;
    PipeCtx px;
    int nF, nB, nC2, nC13;
    BwdEnt e;
};
__global__ void __launch_bounds__(FH_THREADS, 1) update_pipe_ent_kernel(const __grid_constant__ PipeEntArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    int r = (int)blockIdx.x;
    const long long t0 = clock64();
    if (threadIdx.x == 0) prog(a.px, 0, r < a.nF ? 100 : (r < a.nF + a.nB ? 200 : (r < a.nF + a.nB + a.nC2 ? 300 : 400)));
    if (r < a.nF) fwd_role(a.f, a.px, r, a.nF, smem);
    else if (r < a.nF + a.nB) bwd_role<true>(a.b, a.e, a.px, r - a.nF, a.nB, smem);
    else if (r < a.nF + a.nB + a.nC2) dw_role<2>(a.d, a.px, r - a.nF - a.nB, a.nC2, smem);
    else dw_role<3>(a.d, a.px, r - a.nF - a.nB - a.nC2, a.nC13, smem);
    if (threadIdx.x == 0) prog(a.px, 7, (clock64() - t0) >> 10);
}

// ------------------------------------------------------------------------------------------------ loss scale
// S = the power of two that brings max |coef| into [32, 64): fp16 deltas keep their precision (they are ~1e-8 otherwise)
// with a factor 1000 of head-room for the growth through W3 and W2.  scale[0] = S, scale[1] = 1 / S, scale[2] = bits of max.
__global__ void __launch_bounds__(256) absmax_kernel(const float* __restrict__ x, int64_t n, uint32_t* __restrict__ out_bits) {
    float m = 0.0f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) m = fmaxf(m, fabsf(x[i]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.0f && isfinite(m)) atomicMax(out_bits, __float_as_uint(m));
}
// max(|coef| + 1.5 |ecoef|): the bound of the head delta with the entropy bonus (|t_j| <= ln 4 < 1.5, b2048_entropy.cuh)
__global__ void __launch_bounds__(256) absmax_ent_kernel(const float* __restrict__ x, const float* __restrict__ ex, int64_t n,
                                                          uint32_t* __restrict__ out_bits) {
    float m = 0.0f;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        m = fmaxf(m, fmaf(1.5f, fabsf(ex[i]), fabsf(x[i])));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xFFFFFFFFu, m, o));
    if ((threadIdx.x & 31) == 0 && m > 0.0f && isfinite(m)) atomicMax(out_bits, __float_as_uint(m));
}
__global__ void scale_from_max_kernel(float* __restrict__ scale) {
    const float m = __uint_as_float(reinterpret_cast<uint32_t*>(scale)[2]);
    int e = 0;
    if (m > 0.0f) frexpf(m, &e);                   // m = f 2^e, f in [0.5, 1)
    int sh = 6 - e;
    sh = sh > 100 ? 100 : (sh < -100 ? -100 : sh);
    scale[0] = ldexpf(1.0f, sh);
    scale[1] = ldexpf(1.0f, -sh);
}

// ------------------------------------------------------------------------------------------------ host side
struct HpWorkspace {       // byte offsets inside the caller's workspace for a chunk padded to `np` samples
    int64_t h1, h2, dl2, d3t, m1, m2, logits, scale, img, bimg, total;
};
static HpWorkspace hp_workspace(int64_t chunk) {
    HpWorkspace w;
    const int64_t np = (chunk + TC_M - 1) / TC_M * TC_M;
    const int64_t act = np / 64 * ACT_TILE_BYTES, small = np / 64 * SMALL_TILE_BYTES;
    int64_t o = 0;
    w.h1 = o; o += act; w.h2 = o; o += act; w.dl2 = o; o += act;
    w.d3t = o; o += small;
    w.m1 = o; o += np * 32; w.m2 = o; o += np * 32;
    w.logits = o; o += np * 16;
    w.scale = o; o += 1024;
    w.img = o; o += (HP_BYTES + 1023) / 1024 * 1024;
    w.bimg = o; o += (IMG_BYTES + 1023) / 1024 * 1024;
    w.total = o;
    return w;
}

bool backward_hp_supported(const b2048_handle* h, const b2048_mlp_desc* mlp) {
    // log2 observations only: fp16 holds them exactly and the hidden activations stay far below 65504; raw tile values
    // (up to 32768 per input) could overflow the fp16 activations
    return fixed_tc_net(mlp) && mlp->obs_mode == B2048_OBS_LOG2 && h->smem_optin >= PIPE_SMEM && h->smem_optin >= AtbCfg<256>::kSmem;
}

int64_t backward_hp_workspace_bytes(int64_t chunk) { return hp_workspace(chunk).total + 1024; }

static int hp_attrs(b2048_handle* h) {
    if (!(h->attrs & ATTR_HP)) {
        cudaError_t e = cudaFuncSetAttribute(fwd_hp_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, FS_TOTAL);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(fwd_hp_kernel)");
        e = cudaFuncSetAttribute(bwd_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BW_TOTAL);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(bwd_tc_kernel)");
        e = cudaFuncSetAttribute(update_pipe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PIPE_SMEM);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(update_pipe_kernel)");
        e = cudaFuncSetAttribute(bwd_tc_ent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, BW_TOTAL);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(bwd_tc_ent_kernel)");
        e = cudaFuncSetAttribute(update_pipe_ent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, PIPE_SMEM);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(update_pipe_ent_kernel)");
        h->attrs |= ATTR_HP;
    }
    return B2048_OK;
}

static int ensure_hp_image(b2048_handle* h) {
    if (!h->hp_image) {
        cudaError_t e = cudaMalloc(&h->hp_image, (HP_BYTES + 1023) / 1024 * 1024);
        if (e != cudaSuccess) return check_cuda(e, "cudaMalloc(hp_image)");
    }
    return B2048_OK;
}

// b2048_mlp_forward at float32-grade accuracy on the tensor cores: out[n][n_out].  B2048_ERR_UNSUPPORTED (silent) for
// other shapes.
int launch_forward_hp(b2048_handle* h, const b2048_mlp_desc* mlp, const uint64_t* board, float* out, int64_t n, cudaStream_t stream) {
    if (!backward_hp_supported(h, mlp) || n < 4096) return B2048_ERR_UNSUPPORTED;
    { int st = hp_attrs(h); if (st != B2048_OK) return st; }
    { int st = ensure_hp_image(h); if (st != B2048_OK) return st; }
    hp_prepare_kernel<<<64, 256, 0, stream>>>(mlp->W[0], mlp->b[0], mlp->W[1], mlp->b[1], mlp->W[2], mlp->b[2], mlp->dims[3], h->hp_image);
    FwdHpArgs f{};
    f.img = h->hp_image; f.board = board; f.out = out; f.n = n; f.n_out = mlp->dims[3]; f.obs_mode = mlp->obs_mode; f.obs_scale = mlp->obs_log2_scale;
    f.debug_clock = debug_clock_begin(h, B2048_DBG_TC_CLOCKS, stream);
    const int64_t tiles = (n + TC_M - 1) / TC_M;
    const int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
    fwd_hp_kernel<<<grid, FH_THREADS, FS_TOTAL, stream>>>(f);
    int st = check_cuda(cudaGetLastError(), "fwd_hp_kernel launch");
    if (st == B2048_OK && f.debug_clock) {
        long long hb[80];
        if ((st = debug_clock_read(h, hb, 80, stream)) != B2048_OK) return st;
        for (int k = 0; k < 5; ++k) {
            long long* d = hb + 6 * k;
            fprintf(stderr, "[fwd_hp clock] tile %d: wait_d1 %lld epi1 %lld wait_d2 %lld epi2 %lld | to next %lld || mma lane: period %lld, "
                            "layer-2 waits: activations %lld weights %lld\n",
                    k, d[1] - d[0], d[2] - d[1], d[3] - d[2], d[4] - d[3], d[6] - d[0], hb[40 + 4 * (k + 1)], hb[41 + 4 * (k + 1)],
                    hb[42 + 4 * (k + 1)]);
        }
    }
    return st;
}

int launch_loss_scale(const b2048_handle* h, const float* coef, int64_t n, float* scale, cudaStream_t stream, const float* ent_coef) {
    cudaError_t e = cudaMemsetAsync(scale, 0, 16, stream);
    if (e != cudaSuccess) return check_cuda(e, "cudaMemsetAsync(scale)");
    if (ent_coef) absmax_ent_kernel<<<h->num_sms * 4, 256, 0, stream>>>(coef, ent_coef, n, reinterpret_cast<uint32_t*>(scale) + 2);
    else absmax_kernel<<<h->num_sms * 4, 256, 0, stream>>>(coef, n, reinterpret_cast<uint32_t*>(scale) + 2);
    scale_from_max_kernel<<<1, 1, 0, stream>>>(scale);
    return B2048_OK;
}

// The forward stage over `n` samples from `board`, and the backward stage of the same samples (which start at sample c0
// of the caller's arrays), on the workspace `ws` laid out as `w`: shared by the pipelined and the chunked update.
static FwdHpArgs fwd_hp_args(const b2048_mlp_desc* mlp, uint8_t* ws, const HpWorkspace& w, const uint64_t* board, int64_t n) {
    FwdHpArgs f{};
    f.img = ws + w.img; f.board = board; f.out = reinterpret_cast<float*>(ws + w.logits);
    f.h1 = ws + w.h1; f.h2 = ws + w.h2;
    f.m1 = reinterpret_cast<uint64_t*>(ws + w.m1); f.m2 = reinterpret_cast<uint64_t*>(ws + w.m2);
    f.n = n; f.n_out = mlp->dims[3]; f.obs_mode = mlp->obs_mode; f.obs_scale = mlp->obs_log2_scale;
    return f;
}
static BwdArgs bwd_args(const FwdHpArgs& f, uint8_t* ws, const HpWorkspace& w, const uint8_t* mask_flags, const uint8_t* action,
                        const float* coef, int64_t c0, int head_mode, float* const* gW, float* const* gb) {
    BwdArgs b{};
    b.img = ws + w.bimg; b.logits = f.out; b.m1 = f.m1; b.m2 = f.m2; b.board = f.board;
    b.mask_flags = mask_flags ? mask_flags + c0 : nullptr;
    b.action = action ? action + c0 : nullptr;
    b.coef = coef + c0; b.scale = reinterpret_cast<const float*>(ws + w.scale);
    b.dl2 = ws + w.dl2; b.d3t = ws + w.d3t; b.gb3 = gb[2]; b.gW1 = gW[0]; b.gb1 = gb[0];
    b.n = f.n; b.head_mode = head_mode; b.n_out = f.n_out; b.obs_mode = f.obs_mode; b.obs_scale = f.obs_scale;
    return b;
}

// Same contract as the fp32 body of b2048_mlp_backward (grads accumulated, flat layout W_0, b_0, W_1, b_1, ...).
// The whole update of n samples as ONE persistent cooperative launch (see PipeCtx): the SMs are split into forward,
// backward and dW roles; R tile slots of images (R x 206 KB, L2-resident) connect them.
// PA = PipeArgs, or PipeEntArgs (update_pipe_ent_kernel) with ent_coef / ent_sum.
template <class PA>
static int launch_backward_hp_piped(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags, const uint8_t* action,
                                    const float* coef, const b2048_mlp_desc* mlp, float* grads, int64_t n, int head_mode,
                                    uint8_t* ws, int64_t R, cudaStream_t stream, const float* ent_coef, double* ent_sum) {
    constexpr bool kEnt = std::is_same<PA, PipeEntArgs>::value;
    const int n_out = mlp->dims[3];
    const int64_t n_tiles = (n + TC_M - 1) / TC_M;
    const HpWorkspace w = hp_workspace(R * TC_M);
    uint32_t* flags = reinterpret_cast<uint32_t*>(ws + w.total);
    float* scale = reinterpret_cast<float*>(ws + w.scale);
    hp_prepare_kernel<<<64, 256, 0, stream>>>(mlp->W[0], mlp->b[0], mlp->W[1], mlp->b[1], mlp->W[2], mlp->b[2], n_out, ws + w.img);
    bwd_prepare_kernel<<<64, 256, 0, stream>>>(mlp->W[1], mlp->W[2], n_out, ws + w.bimg);
    { int st = launch_loss_scale(h, coef, n, scale, stream, ent_coef); if (st != B2048_OK) return st; }
    cudaError_t e = cudaMemsetAsync(flags, 0, (size_t)n_tiles * 16, stream);
    if (e != cudaSuccess) return check_cuda(e, "cudaMemsetAsync(flags)");
    e = cudaMemsetAsync(ws + w.d3t, 0, (size_t)R * 2 * SMALL_TILE_BYTES, stream);     // rows >= n_out of d3^T stay zero
    if (e != cudaSuccess) return check_cuda(e, "cudaMemsetAsync(d3t)");
    PA a;
    a.px.f_done = flags; a.px.b_done = flags + n_tiles; a.px.c2_done = flags + 2 * n_tiles; a.px.c13_done = flags + 3 * n_tiles;
    a.px.R = R;
    a.px.progress = nullptr;
    if (h->debug & (1u << B2048_DBG_TC_CLOCKS)) {
        for (int i = 0; i < DBG_PROGRESS_WORDS; ++i) h->dbg_progress[i] = -1;
        int* dptr = nullptr;
        e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&dptr), h->dbg_progress, 0);
        if (e != cudaSuccess) return check_cuda(e, "cudaHostGetDevicePointer(progress)");
        a.px.progress = dptr;
    }
    float *gW[B2048_MAX_LAYERS], *gb[B2048_MAX_LAYERS];
    carve_grads(mlp, grads, gW, gb);
    a.f = fwd_hp_args(mlp, ws, w, board, n);
    a.b = bwd_args(a.f, ws, w, mask_flags, action, coef, 0, head_mode, gW, gb);
    a.d.h1 = a.f.h1; a.d.h2 = a.f.h2; a.d.dl2 = a.b.dl2; a.d.d3t = a.b.d3t;
    a.d.gW2 = gW[1]; a.d.gb2 = gb[1]; a.d.gW3 = gW[2]; a.d.inv_scale = scale + 1;
    a.d.n_tiles = n_tiles; a.d.n_out = n_out;
    if constexpr (kEnt) { a.e.ent_coef = ent_coef; a.e.ent_sum = ent_sum; }
    // role split (148 SMs -> 78 / 40 / 16 / 14; swept again after the head of the forward role went from 48 to 32 MMAs): per tile the forward role needs ~12 K cycles, the backward role ~7.5 K, the dW2 role ~4.5 K, the dW3 role ~2.5 K (both bound by ~30 B/clk of L2 -> shared-memory bulk copies per SM)
    const int S = h->num_sms;
    a.nB = (h->pipe_split & 0xFF) ? (h->pipe_split & 0xFF) : (S * 27 + 50) / 100;
    a.nC2 = ((h->pipe_split >> 8) & 0xFF) ? ((h->pipe_split >> 8) & 0xFF) : (S * 11 + 50) / 100;
    a.nC13 = ((h->pipe_split >> 16) & 0xFF) ? ((h->pipe_split >> 16) & 0xFF) : (S * 19 + 100) / 200;   // 14 of 148: its 16 M128 N16 MMAs per tile cost 2.5 K cycles
    a.nF = S - a.nB - a.nC2 - a.nC13;
    if (a.nF < 1 || a.nB < 1 || a.nC2 < 1 || a.nC13 < 1) return fail(B2048_ERR_INVALID, "update pipeline: bad role split");
    void* params[] = {&a};
    const void* kernel = kEnt ? reinterpret_cast<const void*>(update_pipe_ent_kernel) : reinterpret_cast<const void*>(update_pipe_kernel);
    e = cudaLaunchCooperativeKernel(kernel, dim3((unsigned)S), dim3(FH_THREADS), params, (size_t)PIPE_SMEM, stream);
    if (e == cudaSuccess && a.px.progress) {      // debug watchdog: a stuck pipeline is reported and the process ends
        for (int ms = 0; ms < 3000 && cudaStreamQuery(stream) == cudaErrorNotReady; ++ms) {
            struct timespec ts = {0, 1000000};
            nanosleep(&ts, nullptr);
        }
        if (cudaStreamQuery(stream) == cudaErrorNotReady) {
            fprintf(stderr, "[update pipeline] stuck after 3 s; n_tiles %lld R %lld roles F %d B %d dW2 %d dW13 %d\n", (long long)n_tiles,
                    (long long)R, a.nF, a.nB, a.nC2, a.nC13);
            for (int b = 0; b < S; ++b) {
                const int* q = h->dbg_progress + b * 8;
                fprintf(stderr, "  cta %3d role %d: [1] %d [2] %d [3] %d [4] %d [5] %d done %d\n", b, q[0], q[1], q[2], q[3], q[4], q[5], q[7]);
            }
            fflush(stderr);
            _exit(3);
        }
        cudaStreamSynchronize(stream);
        long long tot[4] = {0, 0, 0, 0}, wt[4] = {0, 0, 0, 0};
        int cnt[4] = {0, 0, 0, 0};
        for (int b = 0; b < S; ++b) {
            const int* q = h->dbg_progress + b * 8;
            const int role = q[0] / 100 - 1;
            if (role < 0 || role > 3) continue;
            cnt[role]++; tot[role] += q[7]; wt[role] += q[6] > 0 ? q[6] : 0;
        }
        const char* nm[4] = {"forward", "backward+dW1", "dW2", "dW3"};
        for (int r = 0; r < 4; ++r)
            if (cnt[r]) fprintf(stderr, "[update pipeline] %-13s %3d CTAs: %lld K cycles in the kernel, %lld K of them waiting for flags (per CTA)\n",
                                nm[r], cnt[r], tot[r] / cnt[r], wt[r] / cnt[r]);
    }
    return check_cuda(e, "update_pipe_kernel launch");
}

int launch_backward_hp(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags, const uint8_t* action,
                       const float* coef, const b2048_mlp_desc* mlp, float* grads, int64_t n, int head_mode,
                       uint8_t* workspace, int64_t workspace_bytes, int64_t chunk, cudaStream_t stream, const float* ent_coef,
                       double* ent_sum) {
    { int st = hp_attrs(h); if (st != B2048_OK) return st; }
    const int n_out = mlp->dims[3];
    uint8_t* ws = reinterpret_cast<uint8_t*>(((uintptr_t)workspace + 1023) & ~(uintptr_t)1023);
    {   // large batches: the persistent pipeline with an L2-resident ring of tile slots
        const int64_t n_tiles = (n + TC_M - 1) / TC_M;
        const int64_t Rmax = (h->pipe_split >> 24) ? (int64_t)(h->pipe_split >> 24) * 16 : 288;   // 288 slots x 206 KB = 59 MB of the 126 MB L2
        const int64_t R = n_tiles < Rmax ? n_tiles : Rmax;
        const int64_t need = hp_workspace(R * TC_M).total + n_tiles * 16 + 2048;
        if (!(h->debug & (1u << B2048_DBG_NO_UPDATE_PIPE)) && n_tiles >= 4 * (int64_t)h->num_sms && need <= workspace_bytes) {
            const int st = ent_coef ? launch_backward_hp_piped<PipeEntArgs>(h, board, mask_flags, action, coef, mlp, grads, n, head_mode,
                                                                            ws, R, stream, ent_coef, ent_sum)
                                    : launch_backward_hp_piped<PipeArgs>(h, board, mask_flags, action, coef, mlp, grads, n, head_mode, ws,
                                                                         R, stream, nullptr, nullptr);
            if (st == B2048_OK) return st;
            // the cooperative launch was refused (e.g. the device cannot hold all CTAs at once because it is shared): nothing of
            // the pipeline has run, so the chunked kernel sequence below does the same work
            cudaGetLastError();
        }
    }
    const HpWorkspace w = hp_workspace(chunk);
    float* scale = reinterpret_cast<float*>(ws + w.scale);
    hp_prepare_kernel<<<64, 256, 0, stream>>>(mlp->W[0], mlp->b[0], mlp->W[1], mlp->b[1], mlp->W[2], mlp->b[2], n_out, ws + w.img);
    bwd_prepare_kernel<<<64, 256, 0, stream>>>(mlp->W[1], mlp->W[2], n_out, ws + w.bimg);
    { int st = launch_loss_scale(h, coef, n, scale, stream, ent_coef); if (st != B2048_OK) return st; }
    float *gW[B2048_MAX_LAYERS], *gb[B2048_MAX_LAYERS];
    carve_grads(mlp, grads, gW, gb);
    long long* dbg = debug_clock_begin(h, B2048_DBG_TC_CLOCKS, stream);     // clocks of the first chunk's bwd_tc_kernel
    for (int64_t c0 = 0; c0 < n; c0 += chunk) {
        const int64_t cn = (n - c0) < chunk ? (n - c0) : chunk;
        const int64_t tiles = (cn + TC_M - 1) / TC_M;
        const int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
        const FwdHpArgs f = fwd_hp_args(mlp, ws, w, board + c0, cn);
        fwd_hp_kernel<<<grid, FH_THREADS, FS_TOTAL, stream>>>(f);
        int st = check_cuda(cudaGetLastError(), "fwd_hp_kernel launch");
        if (st != B2048_OK) return st;
        BwdArgs b = bwd_args(f, ws, w, mask_flags, action, coef, c0, head_mode, gW, gb);
        if (c0 == 0) b.debug_clock = dbg;
        cudaError_t e = cudaMemsetAsync(b.d3t, 0, (size_t)tiles * 2 * SMALL_TILE_BYTES, stream);
        if (e != cudaSuccess) return check_cuda(e, "cudaMemsetAsync(d3t)");
        if (ent_coef) {
            BwdEntArgs be;
            be.b = b; be.e.ent_coef = ent_coef + c0; be.e.ent_sum = ent_sum;
            bwd_tc_ent_kernel<<<grid, BW_THREADS, BW_TOTAL, stream>>>(be);
        } else {
            bwd_tc_kernel<<<grid, BW_THREADS, BW_TOTAL, stream>>>(b);
        }
        st = check_cuda(cudaGetLastError(), "bwd_tc_kernel launch");
        if (st != B2048_OK) return st;
        if (b.debug_clock) {
            long long hb[64];
            if ((st = debug_clock_read(h, hb, 64, stream)) != B2048_OK) return st;
            for (int k = 0; k < 5; ++k) {
                long long* d = hb + 8 * k;
                fprintf(stderr, "[bwd_tc clock] tile %d: wait_d5 %lld wait_free %lld epi3 %lld wait_d4 %lld epi4 %lld | to next %lld\n", k,
                        d[1] - d[0], d[2] - d[1], d[3] - d[2], d[4] - d[3], d[5] - d[4], d[8] - d[0]);
            }
        }
        AtbArgs g;
        g.tiles64 = tiles * 2; g.f16 = 1; g.inv_scale = scale + 1;
        // dW2 = H1^T DL2, db2 = column sums of DL2
        g.A = f.h1; g.B = b.dl2; g.C = gW[1]; g.ldm = TC_H; g.ldn = 1; g.n_valid = TC_H; g.colsum = gb[1]; g.colsum_of_b = 1;
        if ((st = launch_atb<256>(h, g, stream)) != B2048_OK) return st;
        // dW3 = H2^T d3
        g.A = f.h2; g.B = b.d3t; g.C = gW[2]; g.ldm = n_out; g.ldn = 1; g.n_valid = n_out; g.colsum = nullptr; g.colsum_of_b = 0;
        if ((st = launch_atb<16>(h, g, stream)) != B2048_OK) return st;
    }
    return B2048_OK;
}

}  // namespace b2
