// b2048_env.cu — environment kernels of libb2048 (sm_100a) and their C entry points.
//
//   K0 build_lut_kernel   Game2048._row_move_left tabulated over all 65,536 rows (game2048.py:120-137)
//   K1 reset_kernel       Game2048.reset + Game2048Env.reset              (game2048.py:26-34, env.py:174-194)
//   K2 step_kernel        fused Game2048.step + Game2048Env.step          (game2048.py:40-70, env.py:197-302)
//      np_seed_kernel / reset_np_kernel / step_np_kernel: the same with the spawns drawn from per-board NumPy streams
//                         (np.random.default_rng(env_seed), b2048_np_rng.cuh) — the reference's own seeded episodes
//      move_kernel        Game2048._move preview                          (game2048.py:158-165)
//      obs_kernel         Game2048Env._preprocess_board                   (env.py:131-150)
//
// Data layout in HBM: structure-of-arrays, one element per board: board u64, score u32, step u32,
// max_exp u8, action u8, reward f32, flags u8.  One thread owns one board; a warp touches 256 B of
// boards, 32 B of actions / flags, 128 B of rewards per step, all fully coalesced.
//
// K2 is bound by instruction issue, not HBM (DESIGN.md): the 192 KB row tables are staged into
// shared memory once per CTA by bulk async copies (TMA engine, cp.async.bulk + mbarrier) that
// overlap the Philox block and the board loads; one persistent 1024-thread CTA per SM then
// grid-strides over the boards.
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>

#include "b2048_internal.h"
#include "b2048_ptx.cuh"
#include "b2048_step_fast.cuh"

namespace b2 {

// ------------------------------------------------------------------------------------------------ K0
__global__ void build_lut_kernel(uint16_t* __restrict__ lut_left, uint8_t* __restrict__ lut_merge) {
    uint32_t row = blockIdx.x * blockDim.x + threadIdx.x;
    if (row >= 65536u) return;
    uint32_t out, merge;
    row_move_left(row, out, merge);
    lut_left[row] = (uint16_t)out;
    lut_merge[row] = (uint8_t)merge;
}

__global__ void build_small_tables_kernel(uint8_t* __restrict__ small) {
    static_assert(B2048_SMALL_BYTES == B2048_TABLES_BYTES - B2048_LUT_BYTES, "small table size mismatch");
    const uint32_t tid = threadIdx.x;
    if (tid < 256u) small_table_entry_agg(tid, reinterpret_cast<AggEntry*>(small + B2048_SMALL_AGG_OFF)[tid]);
    if (tid < 4u) small_table_entry_sel(tid, reinterpret_cast<SelEntry*>(small + B2048_SMALL_SEL_OFF)[tid]);
    if (tid < 64u) small[B2048_SMALL_ACT_OFF + tid] = (uint8_t)small_table_entry_act(tid >> 2, tid & 3u);
}

// ------------------------------------------------------------------------------------------------ K1
__global__ void __launch_bounds__(256) reset_kernel(uint64_t* __restrict__ board, uint32_t* __restrict__ score,
                                                     uint32_t* __restrict__ step, uint8_t* __restrict__ max_exp,
                                                     uint8_t* __restrict__ flags,
                                                     const uint8_t* __restrict__ spawn_replay, int64_t n, uint64_t seed,
                                                     uint64_t gid0, uint32_t t) {
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        Board b;
        if (spawn_replay) {  // the two spawns of Game2048.reset chosen by the host (game2048.py:32-33)
            uint32_t r0 = spawn_replay[2 * i], r1 = spawn_replay[2 * i + 1];
            b = place_kth_empty(Board{0u, 0u}, r0 & 0xFu, (r0 & 0x10u) ? 2u : 1u);
            b = place_kth_empty(b, r1 & 0xFu, (r1 & 0x10u) ? 2u : 1u);
        } else {
            b = reset_board(seed, gid0 + (uint64_t)i, t);
        }
        board[i] = to_u64(b);
        if (score) score[i] = 0u;
        if (step) step[i] = 0u;
        if (max_exp) max_exp[i] = 2u;  // max_tile_seen = 4 (env.py:183)
        if (flags) flags[i] = (uint8_t)legal_mask(b);
    }
}

// ------------------------------------------------------------------------------------------------ NumPy streams
// rng[i] = np.random.default_rng(seeds[i]): one thread per seed (b2048_np_rng.cuh)
__global__ void __launch_bounds__(256) np_seed_kernel(const uint64_t* __restrict__ seeds, b2048_np_rng* __restrict__ rng,
                                                       int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x)
        rng[i] = np::seed(seeds[i]);
}

// Game2048.reset with both spawns drawn from the board's env stream (K1 otherwise)
__global__ void __launch_bounds__(256) reset_np_kernel(uint64_t* __restrict__ board, uint32_t* __restrict__ score,
                                                        uint32_t* __restrict__ step, uint8_t* __restrict__ max_exp,
                                                        uint8_t* __restrict__ flags, b2048_np_rng* __restrict__ env_rng,
                                                        int64_t n) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        b2048_np_rng r = env_rng[i];
        const Board b = np::reset_board(r);
        env_rng[i] = r;
        board[i] = to_u64(b);
        if (score) score[i] = 0u;
        if (step) step[i] = 0u;
        if (max_exp) max_exp[i] = 2u;
        if (flags) flags[i] = (uint8_t)legal_mask(b);
    }
}

// ------------------------------------------------------------------------------------------------ K2
struct StepArgs {
    const uint64_t* board_in;
    uint64_t* board_out;
    uint32_t* score;
    uint32_t* step;
    uint8_t* max_exp;
    const uint8_t* action;
    uint8_t* action_out;
    const uint8_t* flags_in;
    const uint8_t* spawn_replay;
    int32_t* ep_len;   // rollout mode: 0 = episode still running; otherwise frozen (finished at that many steps)
    uint32_t ep_t;     // value stored in ep_len when an episode ends in this call
    int32_t* merge_sum;
    float* reward;
    double* reward64;
    uint8_t* flags;
    float* obs;
    const uint8_t* tables;  // device copy of the row tables
    int64_t n;
    uint64_t seed, gid0;
    uint32_t t;
    b2048_env_cfg cfg;
    PhiloxKeys keys;   // Philox round keys of `seed` (host-computed)
    long long* debug_clock;   // optional phase timestamps of a few CTAs (B2048_STEP_DEBUG_CLOCK), else NULL
};

// Thread 0 stages args.tables into shared memory with bulk copies that complete on `mbar` (phase 0): the small tables
// first (needed first, kSmall only), then the row tables in 32 KB pieces.  Ends with every thread past the barrier's
// initialisation, so any thread may wait on it.  `args` is taken by reference: a by-value table pointer costs
// step_fast_n_kernel two registers.
template <bool kSmall, class Args>
__device__ __forceinline__ void stage_tables(uint8_t* smem, const Args& args, uint64_t* mbar) {
    const uint32_t bar = s_u32(mbar);
    if (threadIdx.x == 0) {
        mbar_init(bar, 1);
        mbar_init_fence();
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        mbar_expect_tx(bar, kSmall ? (uint32_t)B2048_TABLES_BYTES : (uint32_t)B2048_LUT_BYTES);
        if (kSmall) bulk_load(s_u32(smem + B2048_LUT_BYTES), args.tables + B2048_LUT_BYTES, (uint32_t)B2048_SMALL_BYTES, bar);
        bulk_load_chunked<32768u>(s_u32(smem), args.tables, (uint32_t)B2048_LUT_BYTES, bar);
    }
}

// 128-bit coalesced observation stores for raw / log2: lane l of store round s writes row (l & 3) of
// the board held by lane 8s + (l >> 2), so consecutive lanes write consecutive 16-byte chunks.
__device__ __forceinline__ void store_obs16(float* __restrict__ obs, Board nb, int64_t warp_base, int64_t n, int lane,
                                            int obs_mode, float scale) {
#pragma unroll
    for (int s = 0; s < 4; ++s) {
        int src = 8 * s + (lane >> 2);
        uint32_t lo = __shfl_sync(0xFFFFFFFFu, nb.lo, src);
        uint32_t hi = __shfl_sync(0xFFFFFFFFu, nb.hi, src);
        int row = lane & 3;
        uint32_t w = (row & 2) ? hi : lo;
        uint32_t r16 = (w >> (16 * (row & 1))) & 0xFFFFu;
        float v[4];
        encode_row(r16, obs_mode, scale, v);
        int64_t bi = warp_base + src;
        if (bi < n) {
            float4 q = make_float4(v[0], v[1], v[2], v[3]);
            *reinterpret_cast<float4*>(obs + bi * 16 + row * 4) = q;
        }
    }
}

// onehot [16][17] float32 per board = 68 float4: the warp writes board after board, 128-bit per lane
__device__ __forceinline__ void store_obs_onehot(float* __restrict__ obs, Board nb, int64_t warp_base, int64_t n,
                                                 int lane) {
    for (int j = 0; j < 32; ++j) {
        int64_t bi = warp_base + j;
        if (bi >= n) break;  // warp-uniform
        uint32_t lo = __shfl_sync(0xFFFFFFFFu, nb.lo, j);
        uint32_t hi = __shfl_sync(0xFFFFFFFFu, nb.hi, j);
        uint64_t b = (uint64_t)lo | ((uint64_t)hi << 32);
        float4* dst = reinterpret_cast<float4*>(obs + bi * 272);
#pragma unroll
        for (int q0 = 0; q0 < 96; q0 += 32) {
            int q = q0 + lane;
            if (q < 68) {
                float v[4];
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    int f = 4 * q + u;
                    int cell = f / 17, ch = f - 17 * cell;
                    int e = (int)((b >> (4 * cell)) & 0xFull);
                    v[u] = (e == ch) ? 1.0f : 0.0f;
                }
                dst[q] = make_float4(v[0], v[1], v[2], v[3]);
            }
        }
    }
}

// The body of step_kernel and of its reference-seeded variant step_np_kernel (kNp: spawns from the boards' NumPy env
// streams env_rng, advanced in place; buffer actions, no auto-reset).
template <bool kSmemLut, int kThreads, bool kNp>
__device__ __forceinline__ void step_loop(const StepArgs& args, b2048_np_rng* env_rng) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t mbar;

    const int tid = threadIdx.x;
    __builtin_assume(tid < kThreads);   // the launch bound, which the kernel's range analysis does not see through the inlined body
    const int lane = tid & 31;
    const uint16_t* lut_left;
    const uint8_t* lut_merge;

    if (kSmemLut) {
        // Stage both row tables (192 KB) into shared memory with the bulk-copy engine; completion is
        // signalled on an mbarrier so the copy overlaps the first iteration's loads and Philox block.
        stage_tables<false>(smem, args, &mbar);
        lut_left = reinterpret_cast<const uint16_t*>(smem);
        lut_merge = smem + B2048_LUT_LEFT_BYTES;
    } else {
        lut_left = reinterpret_cast<const uint16_t*>(args.tables);
        lut_merge = args.tables + B2048_LUT_LEFT_BYTES;
    }

    const b2048_env_cfg& cfg = args.cfg;
    StepOpts opt;
    opt.track_step = args.step != nullptr;
    opt.track_max = args.max_exp != nullptr;
    opt.want_sum = cfg.reward_mode == B2048_REWARD_SUM || args.score != nullptr || args.merge_sum != nullptr;

    bool lut_ready = !kSmemLut;
    const int64_t stride = (int64_t)gridDim.x * kThreads;
    for (int64_t base = (int64_t)blockIdx.x * kThreads; base < args.n; base += stride) {
        const int64_t i = base + tid;
        const bool valid = i < args.n;
        StepIO io;
        io.board = Board{0u, 0u};
        io.score = 0u;
        io.step = 0u;
        io.max_exp = 2u;
        io.action = 0u;
        io.mask_in = 0u;
        io.have_mask_in = args.flags_in != nullptr;
        io.replay = 0u;
        if (valid) {
            if (args.spawn_replay) io.replay = args.spawn_replay[i];
            io.board = make_board(args.board_in[i]);
            if (args.score) io.score = args.score[i];
            if (args.step) io.step = args.step[i];
            if (args.max_exp) io.max_exp = args.max_exp[i];
            if (cfg.action_mode == B2048_ACT_BUFFER) io.action = args.action[i];
            if (args.flags_in) io.mask_in = args.flags_in[i];
        }
        if (!lut_ready) {
            // all threads wait on phase 0 of the table barrier (returns immediately once complete)
            mbar_wait(s_u32(&mbar), 0);
            lut_ready = true;
        }
        bool frozen = false;
        Board board_before = io.board;
        if (args.ep_len && valid) frozen = args.ep_len[i] != 0;
        b2048_np_rng rng;
        if constexpr (kNp) {
            if (valid && !frozen) rng = env_rng[i];
        }
        step_one<decltype(lut_left), decltype(lut_merge), kNp>(io, cfg, opt, args.seed, args.gid0 + (uint64_t)i, args.t,
                                                              lut_left, lut_merge, &rng, valid && !frozen);
        if (valid && frozen) {
            // finished episode of a run-to-termination rollout: pass the terminal state through untouched
            uint32_t m = legal_mask(board_before);
            uint32_t f = args.flags_in ? (uint32_t)args.flags_in[i]
                                       : (m | ((m == 0u && (board_before.lo | board_before.hi) != 0u) ? B2048_F_DONE : 0u));
            args.board_out[i] = to_u64(board_before);
            if (args.action_out) args.action_out[i] = 0;
            if (args.merge_sum) args.merge_sum[i] = 0;
            if (args.reward) args.reward[i] = 0.0f;
            if (args.reward64) args.reward64[i] = 0.0;
            args.flags[i] = (uint8_t)(f & ~B2048_F_CHANGED);
            io.board = board_before;
        } else if (valid) {
            if (args.ep_len && (io.flags & (B2048_F_DONE | B2048_F_TRUNC))) args.ep_len[i] = (int32_t)args.ep_t;
            args.board_out[i] = to_u64(io.board);
            if (args.score) args.score[i] = io.score;
            if (args.step) args.step[i] = io.step;
            if (args.max_exp) args.max_exp[i] = (uint8_t)io.max_exp;
            if (args.action_out) args.action_out[i] = (uint8_t)io.action_played;
            if (args.merge_sum) args.merge_sum[i] = io.merge_sum;
            if (args.reward) args.reward[i] = (float)io.reward;
            if (args.reward64) args.reward64[i] = io.reward;
            args.flags[i] = (uint8_t)io.flags;
            if constexpr (kNp) {
                if (io.flags & B2048_F_CHANGED) env_rng[i] = rng;   // only a changed board drew a spawn
            }
        }
        if (args.obs != nullptr && cfg.obs_mode != B2048_OBS_NONE) {
            const int64_t warp_base = base + (tid & ~31);
            if (cfg.obs_mode == B2048_OBS_ONEHOT) store_obs_onehot(args.obs, io.board, warp_base, args.n, lane);
            else store_obs16(args.obs, io.board, warp_base, args.n, lane, cfg.obs_mode, cfg.obs_log2_scale);
        }
    }
}

template <bool kSmemLut, int kThreads>
__global__ void __launch_bounds__(kThreads, kSmemLut ? 1 : 2) step_kernel(const __grid_constant__ StepArgs args) {
    step_loop<kSmemLut, kThreads, false>(args, nullptr);
}

template <bool kSmemLut, int kThreads>
__global__ void __launch_bounds__(kThreads, kSmemLut ? 1 : 2) step_np_kernel(const __grid_constant__ StepArgs args,
                                                                              b2048_np_rng* __restrict__ env_rng) {
    step_loop<kSmemLut, kThreads, true>(args, env_rng);
}

// ------------------------------------------------------------------------------------------------ K2 (fast path)
// Same contract as step_kernel for the common configuration (see b2048_step_fast.cuh); all tables in
// shared memory, brought in by one mbarrier-tracked bulk copy per CTA.
// kPlain: no rollout bookkeeping and no optional outputs (ep_len, action_out, merge_sum, debug clocks all NULL), the
// previous legal masks supplied, fewer than 2^31 boards — the configuration of every large env-only batch.  The loop
// then carries no frozen-episode logic, no predicated-off stores, one wait for the tables before the loop and 32-bit
// indices (one IMAD.WIDE per address instead of a LEA pair): the kernel is bound by issue slots, not by memory.
template <int kAct, bool kTrack, bool kPlain>
__global__ void __launch_bounds__(1024, 1) step_fast_kernel(const __grid_constant__ StepArgs args) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t mbar;
    const int tid = threadIdx.x;
    const bool dbg = args.debug_clock != nullptr && tid == 0 && (blockIdx.x == 0 || blockIdx.x == 147);
    long long* dc = dbg ? args.debug_clock + (blockIdx.x == 0 ? 0 : 16) : nullptr;
    int dci = 0;
    if (dbg) { dc[dci++] = (long long)globaltimer(); dc[dci++] = clock64(); }
    // Programmatic dependent launch (no-ops when the launch does not carry the attribute): the NEXT launch in the
    // stream may start placing its CTAs as soon as SMs free up, so its barrier set-up and its 194 KB table staging run
    // under this launch's tail; it reads or writes nothing a previous launch touched before its own griddepcontrol.wait.
    pdl_launch_dependents();
    stage_tables<true>(smem, args, &mbar);
    FastTables T;
    T.left = reinterpret_cast<const uint16_t*>(smem);
    T.merge = smem + B2048_LUT_LEFT_BYTES;
    T.agg = reinterpret_cast<const AggEntry*>(smem + B2048_LUT_BYTES + B2048_SMALL_AGG_OFF);
    T.sel = reinterpret_cast<const SelEntry*>(smem + B2048_LUT_BYTES + B2048_SMALL_SEL_OFF);
    T.act = smem + B2048_LUT_BYTES + B2048_SMALL_ACT_OFF;
    // everything above touched only the static tables; the boards may have been written by the previous launch
    pdl_wait();

    const b2048_env_cfg& cfg = args.cfg;
    if constexpr (kPlain) {
        const uint32_t n = (uint32_t)args.n, stride = gridDim.x * 1024u;
        uint32_t i = blockIdx.x * 1024u + (uint32_t)tid;
        // software pipeline: the next iteration's inputs are requested before the current board is processed
        uint2 bw_next = make_uint2(0u, 0u);
        uint32_t act_next = 0u, fin_next = 0u, score_next = 0u, step_next = 0u, max_next = 2u;
        auto request = [&](uint32_t k) {
            bw_next = *reinterpret_cast<const uint2*>(args.board_in + k);
            if (kAct == B2048_ACT_BUFFER) act_next = args.action[k];
            else if (kAct != B2048_ACT_RANDOM_ANY) fin_next = args.flags_in[k];
            if (kTrack) { score_next = args.score[k]; step_next = args.step[k]; max_next = args.max_exp[k]; }
        };
        if (i < n) request(i);
        // the Philox block of the first board is computed while the tables arrive; later ones at the end of the
        // previous iteration (same instruction count, the first one is off the staging's critical path)
        Rand4 rnd = stream_keyed(args.keys, args.gid0 + (uint64_t)i, args.t, B2048_DOM_STEP);
        mbar_wait(s_u32(&mbar), 0);   // the tables have to be in shared memory before the first lookup
        for (; i < n; i += stride) {
            FastIO io;
            io.lo = bw_next.x; io.hi = bw_next.y;
            io.score = score_next; io.step = step_next; io.max_exp = max_next;
            io.action = act_next; io.mask_in = fin_next;
            const uint32_t inext = i + stride;
            if (inext < n) request(inext);
            step_fast_rnd<kAct, kTrack, false>(io, cfg, rnd, args.keys, args.gid0 + (uint64_t)i, args.t, T);   // kPlain: unshaped rewards
            *reinterpret_cast<uint2*>(args.board_out + i) = make_uint2(io.lo, io.hi);
            if (kTrack) { args.score[i] = io.score; args.step[i] = io.step; args.max_exp[i] = (uint8_t)io.max_exp; }
            args.reward[i] = io.reward;
            args.flags[i] = (uint8_t)io.flags;
            if (inext < n) rnd = stream_keyed(args.keys, args.gid0 + (uint64_t)inext, args.t, B2048_DOM_STEP);
        }
        return;
    }
    bool ready = false;
    const int64_t stride = (int64_t)gridDim.x * 1024;
    int64_t i = (int64_t)blockIdx.x * 1024 + tid;
    // software pipeline: the next iteration's board / action / mask are requested before the current
    // board is processed, so the ~800-cycle HBM latency is off the critical path of every iteration
    uint2 bw_next = make_uint2(0u, 0u);
    uint32_t act_next = 0u, fin_next = 0u;
    if (i < args.n) {
        bw_next = *reinterpret_cast<const uint2*>(args.board_in + i);
        if (kAct == B2048_ACT_BUFFER) act_next = args.action[i];
        if (args.flags_in) fin_next = args.flags_in[i];
    }
    for (; i < args.n; i += stride) {
        FastIO io;
        const uint2 bw = bw_next;
        const uint32_t fin = fin_next;
        io.lo = bw.x; io.hi = bw.y;
        io.score = 0u; io.step = 0u; io.max_exp = 2u; io.mask_in = 0u;
        io.action = act_next;
        const int64_t inext = i + stride;
        if (inext < args.n) {
            bw_next = *reinterpret_cast<const uint2*>(args.board_in + inext);
            if (kAct == B2048_ACT_BUFFER) act_next = args.action[inext];
            if (args.flags_in) fin_next = args.flags_in[inext];
        }
        if (kTrack) { io.score = args.score[i]; io.step = args.step[i]; io.max_exp = args.max_exp[i]; }
        if (kAct == B2048_ACT_RANDOM_LEGAL || kAct == B2048_ACT_PRIORITY)
            io.mask_in = args.flags_in ? fin : legal_mask(Board{io.lo, io.hi});
        bool frozen = false;
        if (args.ep_len) frozen = args.ep_len[i] != 0;
        if (!ready) {
            mbar_wait(s_u32(&mbar), 0);
            ready = true;
            if (dbg) dc[dci++] = clock64();
        }
        if (frozen) {   // finished episode of a run-to-termination rollout: pass through (see step_kernel)
            uint32_t m = legal_mask(Board{io.lo, io.hi});
            uint32_t f = args.flags_in ? fin : (m | ((m == 0u && (io.lo | io.hi) != 0u) ? B2048_F_DONE : 0u));
            *reinterpret_cast<uint2*>(args.board_out + i) = bw;
            if (args.action_out) args.action_out[i] = 0;
            if (args.merge_sum) args.merge_sum[i] = 0;
            args.reward[i] = 0.0f;
            args.flags[i] = (uint8_t)(f & ~B2048_F_CHANGED);
            continue;
        }
        step_fast<kAct, kTrack>(io, cfg, args.keys, args.seed, args.gid0 + (uint64_t)i, args.t, T);
        if (args.ep_len && (io.flags & (B2048_F_DONE | B2048_F_TRUNC))) args.ep_len[i] = (int32_t)args.ep_t;
        *reinterpret_cast<uint2*>(args.board_out + i) = make_uint2(io.lo, io.hi);
        if (kTrack) { args.score[i] = io.score; args.step[i] = io.step; args.max_exp[i] = (uint8_t)io.max_exp; }
        if (args.action_out) args.action_out[i] = (uint8_t)io.action;
        if (args.merge_sum) args.merge_sum[i] = io.merge_sum;
        args.reward[i] = io.reward;
        args.flags[i] = (uint8_t)io.flags;
        if (dbg && dci < 12) dc[dci++] = clock64();
    }
    if (dbg) { const unsigned long long gt = globaltimer(); dc[14] = clock64(); dc[15] = (long long)gt; }
}

// Launched with cudaLaunchAttributeProgrammaticStreamSerialization (programmatic dependent launch): when the previous
// kernel in the stream is another step launch, this one's prologue (barrier set-up, table staging) overlaps its tail
// instead of waiting for the grid to drain and the launch to travel; after any other kernel it degrades to plain
// stream order (griddepcontrol.wait returns once that kernel has completed).
template <int kAct, bool kTrack, bool kPlain>
static cudaError_t launch_fast_one(int grid, size_t smem, cudaStream_t s, const StepArgs& a, bool pdl) {
    cudaLaunchConfig_t lc = {};
    lc.gridDim = dim3((unsigned)grid); lc.blockDim = dim3(1024); lc.dynamicSmemBytes = smem; lc.stream = s;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    lc.attrs = at; lc.numAttrs = pdl ? 1u : 0u;
    return cudaLaunchKernelEx(&lc, step_fast_kernel<kAct, kTrack, kPlain>, a);
}
template <int kAct>
static cudaError_t launch_fast(bool track, int grid, size_t smem, cudaStream_t s, const StepArgs& a, bool pdl) {
    const bool plain = a.ep_len == nullptr && a.action_out == nullptr && a.merge_sum == nullptr && a.debug_clock == nullptr &&
                       (kAct == B2048_ACT_BUFFER || kAct == B2048_ACT_RANDOM_ANY || a.flags_in != nullptr) &&
                       a.n < ((int64_t)1 << 31) - (int64_t)grid * 1024 &&
                       // the plain specialisation compiles the reward-shaping terms out (step_fast_rnd<.., kShaped = false>)
                       !cfg_is_shaped(a.cfg);
    if (plain) return track ? launch_fast_one<kAct, true, true>(grid, smem, s, a, pdl) : launch_fast_one<kAct, false, true>(grid, smem, s, a, pdl);
    return track ? launch_fast_one<kAct, true, false>(grid, smem, s, a, pdl) : launch_fast_one<kAct, false, false>(grid, smem, s, a, pdl);
}

// ------------------------------------------------------------------------------------------------ multi-step
// n_steps consecutive steps of a device-side action mode in ONE launch: each thread keeps its board, counters and legal
// mask in registers across the steps and writes only the final state — no per-step HBM traffic, no per-step launch
// or table staging.  Same result as n_steps single-step launches with t, t + 1, ... (tested bit for bit).
struct StepNArgs {
    uint64_t* board;
    uint32_t* score;
    uint32_t* step;
    uint8_t* max_exp;
    uint8_t* flags;          // in (low 4 bits = legal mask of board, when flags_valid) / out (flags of the last step)
    float* reward_last;      // optional: reward of the last step
    float* reward_sum;       // optional: += float32 sum of the per-step rewards (step order)
    int32_t* episodes;       // optional: += number of steps that terminated or truncated an episode
    const uint8_t* tables;
    int64_t n;
    int32_t n_steps, flags_valid;
    uint64_t seed, gid0;
    uint32_t t;
    b2048_env_cfg cfg;
    PhiloxKeys keys;
};

template <int kAct, bool kTrack, bool kShaped>
__global__ void __launch_bounds__(1024, 1) step_fast_n_kernel(const __grid_constant__ StepNArgs args) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ uint64_t mbar;
    const int tid = threadIdx.x;
    stage_tables<true>(smem, args, &mbar);
    FastTables T;
    T.left = reinterpret_cast<const uint16_t*>(smem);
    T.merge = smem + B2048_LUT_LEFT_BYTES;
    T.agg = reinterpret_cast<const AggEntry*>(smem + B2048_LUT_BYTES + B2048_SMALL_AGG_OFF);
    T.sel = reinterpret_cast<const SelEntry*>(smem + B2048_LUT_BYTES + B2048_SMALL_SEL_OFF);
    T.act = smem + B2048_LUT_BYTES + B2048_SMALL_ACT_OFF;
    const b2048_env_cfg& cfg = args.cfg;
    bool ready = false;
    const int64_t stride = (int64_t)gridDim.x * 1024;
    for (int64_t i = (int64_t)blockIdx.x * 1024 + tid; i < args.n; i += stride) {
        FastIO io;
        const uint2 bw = *reinterpret_cast<const uint2*>(args.board + i);
        io.lo = bw.x; io.hi = bw.y;
        io.score = 0u; io.step = 0u; io.max_exp = 2u; io.action = 0u;
        if (kTrack) { io.score = args.score[i]; io.step = args.step[i]; io.max_exp = args.max_exp[i]; }
        io.mask_in = args.flags_valid ? (uint32_t)args.flags[i] : legal_mask(Board{io.lo, io.hi});
        io.flags = io.mask_in;
        io.reward = 0.0f;
        if (!ready) {
            mbar_wait(s_u32(&mbar), 0);
            ready = true;
        }
        float rsum = 0.0f;
        int32_t eps = 0;
        const uint64_t gid = args.gid0 + (uint64_t)i;
        for (int32_t k = 0; k < args.n_steps; ++k) {
            io.mask_in = io.flags & 0xFu;          // the flags of a step carry the legal mask of the board it returns
            step_fast<kAct, kTrack, kShaped>(io, cfg, args.keys, args.seed, gid, args.t + (uint32_t)k, T);
            rsum += io.reward;
            eps += (io.flags & (B2048_F_DONE | B2048_F_TRUNC)) ? 1 : 0;
        }
        *reinterpret_cast<uint2*>(args.board + i) = make_uint2(io.lo, io.hi);
        if (kTrack) { args.score[i] = io.score; args.step[i] = io.step; args.max_exp[i] = (uint8_t)io.max_exp; }
        args.flags[i] = (uint8_t)io.flags;
        if (args.reward_last) args.reward_last[i] = io.reward;
        if (args.reward_sum) args.reward_sum[i] += rsum;
        if (args.episodes) args.episodes[i] += eps;
    }
}

// ------------------------------------------------------------------------------------------------ previews
__global__ void __launch_bounds__(256) move_kernel(const uint64_t* __restrict__ board_in, uint64_t* __restrict__ board_out,
                                                    const uint8_t* __restrict__ action, int32_t* __restrict__ merge_sum,
                                                    uint8_t* __restrict__ merge_info, uint8_t* __restrict__ flags,
                                                    const uint8_t* __restrict__ tables, int64_t n) {
    const uint16_t* lut_left = reinterpret_cast<const uint16_t*>(tables);
    const uint8_t* lut_merge = tables + B2048_LUT_LEFT_BYTES;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        Board b = make_board(board_in[i]);
        MoveResult mv = move_board(b, action[i] & 3u, lut_left, lut_merge);
        MergeStats ms = merge_stats(mv.merge, true, false);
        uint32_t mask = legal_mask(mv.board);
        bool changed = (mv.board.lo != b.lo) | (mv.board.hi != b.hi);
        bool done = (mask == 0u) & ((mv.board.lo | mv.board.hi) != 0u);
        board_out[i] = to_u64(mv.board);
        if (merge_sum) merge_sum[i] = (int32_t)ms.sum;
        if (merge_info) *reinterpret_cast<uint32_t*>(merge_info + 4 * i) = mv.merge;
        if (flags)
            flags[i] = (uint8_t)(mask | (changed ? B2048_F_CHANGED : 0u) | (done ? B2048_F_DONE : 0u) |
                                 (ms.overflow ? B2048_F_OVERFLOW : 0u));
    }
}

__global__ void __launch_bounds__(256) obs_kernel(const uint64_t* __restrict__ board, float* __restrict__ obs, int obs_mode,
                                                   float scale, int64_t n) {
    const int lane = threadIdx.x & 31;
    int64_t stride = (int64_t)gridDim.x * blockDim.x;
    for (int64_t base = (int64_t)blockIdx.x * blockDim.x; base < n; base += stride) {
        int64_t i = base + threadIdx.x;
        Board b = i < n ? make_board(board[i]) : Board{0u, 0u};
        int64_t warp_base = base + (threadIdx.x & ~31);
        if (obs_mode == B2048_OBS_ONEHOT) store_obs_onehot(obs, b, warp_base, n, lane);
        else store_obs16(obs, b, warp_base, n, lane, obs_mode, scale);
    }
}

// ------------------------------------------------------------------------------------------------ D4 symmetries
// Game2048Env.get_symmetries (src/env.py:317-397) / _augment_trajectories (src/reinforce_agent.py:773-808) on packed
// boards: variant v of (board, action, mask) is a nibble permutation of the board, a relabelling of the action and
// a permutation of the four mask bits.  Variants in the reference's order: identity + three counter-clockwise
// quarter turns (np.rot90 k=1, action (a-1)%4, mask roll -1), then the same four for the left-right mirror
// (np.fliplr, actions 1 <-> 3, mask [0,3,2,1]).
struct SymVariant {
    uint64_t perm;    // nibble i = source cell of destination cell i
    uint32_t amap;    // bits 2a..2a+1 = new label of action a
    uint32_t mperm;   // bits 2i..2i+1 = source mask bit of destination mask bit i
};
__constant__ SymVariant kSym[8] = {
    {0xFEDCBA9876543210ull, 0xE4u, 0xE4u}, {0xC840D951EA62FB73ull, 0x93u, 0x39u},
    {0x0123456789ABCDEFull, 0x4Eu, 0x4Eu}, {0x37BF26AE159D048Cull, 0x39u, 0x93u},
    {0xCDEF89AB45670123ull, 0x6Cu, 0x6Cu}, {0xFB73EA62D951C840ull, 0x1Bu, 0x1Bu},
    {0x32107654BA98FEDCull, 0xC6u, 0xC6u}, {0x048C159D26AE37BFull, 0xB1u, 0xB1u},
};

// out arrays are [rows][8 * n]: variant v of element (r, i) goes to r * 8n + v * n + i, i.e. the batch axis becomes
// eight concatenated copies (what update_batch sees after _augment_trajectories).
__global__ void __launch_bounds__(256) symmetries_kernel(const uint64_t* __restrict__ board, const uint8_t* __restrict__ flags,
                                                          const uint8_t* __restrict__ action, uint64_t* __restrict__ board_out,
                                                          uint8_t* __restrict__ flags_out, uint8_t* __restrict__ action_out,
                                                          int64_t rows, int64_t n) {
    const int64_t total = rows * n;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t r = e / n, i = e - r * n;
        const uint64_t b = board ? board[e] : 0ull;
        const uint32_t f = flags ? flags[e] : 0u, a = action ? (action[e] & 3u) : 0u;
#pragma unroll
        for (int v = 0; v < 8; ++v) {
            const SymVariant sv = kSym[v];
            const int64_t o = r * 8 * n + (int64_t)v * n + i;
            if (board_out) {
                uint64_t nb = 0;
#pragma unroll
                for (int c = 0; c < 16; ++c) nb |= ((b >> (4 * (uint32_t)((sv.perm >> (4 * c)) & 0xFull))) & 0xFull) << (4 * c);
                board_out[o] = nb;
            }
            if (flags_out) {
                uint32_t nf = f & 0xF0u;
#pragma unroll
                for (int k = 0; k < 4; ++k) nf |= ((f >> ((sv.mperm >> (2 * k)) & 3u)) & 1u) << k;
                flags_out[o] = (uint8_t)nf;
            }
            if (action_out) action_out[o] = (uint8_t)((sv.amap >> (2 * a)) & 3u);
        }
    }
}

static int grid_for(int64_t n, int threads, int num_sms, int per_sm) {
    int64_t blocks = (n + threads - 1) / threads;
    int64_t cap = (int64_t)num_sms * per_sm;
    if (blocks > cap) blocks = cap;
    if (blocks < 1) blocks = 1;
    return (int)blocks;
}

}  // namespace b2

// ================================================================================================ C ABI
using namespace b2;

extern "C" int b2048_create(b2048_handle** out) {
    B2_REQUIRE(out != nullptr, "b2048_create: out is NULL");
    b2048_handle* h = new b2048_handle();   // value-initialised: no buffers yet, no attributes set, every debug option off
    B2_CUDA(cudaGetDevice(&h->device));
    B2_CUDA(cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, h->device));
    B2_CUDA(cudaDeviceGetAttribute(&h->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
    B2_CUDA(cudaMalloc(&h->d_tables, B2048_TABLES_BYTES));
    build_lut_kernel<<<256, 256>>>(reinterpret_cast<uint16_t*>(h->d_tables), h->d_tables + B2048_LUT_LEFT_BYTES);
    build_small_tables_kernel<<<1, 256>>>(h->d_tables + B2048_LUT_BYTES);
    B2_CUDA(cudaGetLastError());
    B2_CUDA(cudaDeviceSynchronize());
    if (h->smem_optin >= B2048_LUT_BYTES) {
        B2_CUDA(cudaFuncSetAttribute(step_kernel<true, 1024>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     B2048_LUT_BYTES));
        B2_CUDA(cudaFuncSetAttribute(step_np_kernel<true, 1024>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                     B2048_LUT_BYTES));
    }
    if (h->smem_optin >= B2048_TABLES_BYTES) {
#define B2_SET(A, TR)                                                                                                       \
    B2_CUDA(cudaFuncSetAttribute(step_fast_kernel<A, TR, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, B2048_TABLES_BYTES)); \
    B2_CUDA(cudaFuncSetAttribute(step_fast_kernel<A, TR, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, B2048_TABLES_BYTES))
        B2_SET(B2048_ACT_BUFFER, true); B2_SET(B2048_ACT_BUFFER, false);
        B2_SET(B2048_ACT_RANDOM_LEGAL, true); B2_SET(B2048_ACT_RANDOM_LEGAL, false);
        B2_SET(B2048_ACT_RANDOM_ANY, true); B2_SET(B2048_ACT_RANDOM_ANY, false);
        B2_SET(B2048_ACT_PRIORITY, true); B2_SET(B2048_ACT_PRIORITY, false);
#define B2_SET_N(A, TR)                                                                                                               \
    do {                                                                                                                              \
        B2_CUDA(cudaFuncSetAttribute(step_fast_n_kernel<A, TR, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, B2048_TABLES_BYTES)); \
        B2_CUDA(cudaFuncSetAttribute(step_fast_n_kernel<A, TR, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, B2048_TABLES_BYTES));  \
    } while (0)
        B2_SET_N(B2048_ACT_RANDOM_LEGAL, true); B2_SET_N(B2048_ACT_RANDOM_LEGAL, false);
        B2_SET_N(B2048_ACT_RANDOM_ANY, true); B2_SET_N(B2048_ACT_RANDOM_ANY, false);
        B2_SET_N(B2048_ACT_PRIORITY, true); B2_SET_N(B2048_ACT_PRIORITY, false);
#undef B2_SET_N
#undef B2_SET
    }
    *out = h;
    return B2048_OK;
}

extern "C" int b2048_destroy(b2048_handle* h) {
    if (!h) return B2048_OK;
    cudaFree(h->d_tables);
    if (h->tc_image) cudaFree(h->tc_image);
    if (h->hp_image) cudaFree(h->hp_image);
    if (h->gen_image) cudaFree(h->gen_image);
    if (h->dbg_clock) cudaFree(h->dbg_clock);
    if (h->dbg_progress) cudaFreeHost(h->dbg_progress);
    delete h;
    return B2048_OK;
}

extern "C" int b2048_get_row_lut(b2048_handle* h, uint16_t* lut_left_host, uint8_t* lut_merge_host) {
    B2_REQUIRE(h != nullptr, "b2048_get_row_lut: handle is NULL");
    if (lut_left_host) B2_CUDA(cudaMemcpy(lut_left_host, h->d_tables, B2048_LUT_LEFT_BYTES, cudaMemcpyDeviceToHost));
    if (lut_merge_host)
        B2_CUDA(cudaMemcpy(lut_merge_host, h->d_tables + B2048_LUT_LEFT_BYTES, B2048_LUT_MERGE_BYTES,
                           cudaMemcpyDeviceToHost));
    return B2048_OK;
}

extern "C" int b2048_reset_many(b2048_handle* h, uint64_t* board, uint32_t* score, uint32_t* step, uint8_t* max_exp,
                                uint8_t* flags, const uint8_t* spawn_replay, int64_t n, uint64_t seed, uint64_t gid0,
                                uint32_t t, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_reset_many: handle is NULL");
    B2_REQUIRE(n >= 0, "b2048_reset_many: n < 0");
    B2_REQUIRE(board != nullptr || n == 0, "b2048_reset_many: board is NULL");
    if (n == 0) return B2048_OK;
    reset_kernel<<<grid_for(n, 256, h->num_sms, 8), 256, 0, (cudaStream_t)stream>>>(board, score, step, max_exp, flags,
                                                                                   spawn_replay, n, seed, gid0, t);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_np_rng_seed(const uint64_t* seeds, b2048_np_rng* rng, int64_t n, void* stream) {
    B2_REQUIRE(n >= 0, "b2048_np_rng_seed: n < 0");
    if (n == 0) return B2048_OK;
    B2_REQUIRE(seeds && rng, "b2048_np_rng_seed: seeds / rng is NULL");
    const int64_t blocks = (n + 255) / 256;
    np_seed_kernel<<<(unsigned)(blocks < 65536 ? blocks : 65536), 256, 0, (cudaStream_t)stream>>>(seeds, rng, n);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_reset_many_np(b2048_handle* h, uint64_t* board, uint32_t* score, uint32_t* step, uint8_t* max_exp,
                                   uint8_t* flags, b2048_np_rng* env_rng, int64_t n, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_reset_many_np: handle is NULL");
    B2_REQUIRE(n >= 0, "b2048_reset_many_np: n < 0");
    if (n == 0) return B2048_OK;
    B2_REQUIRE(board && env_rng, "b2048_reset_many_np: board / env_rng is NULL");
    reset_np_kernel<<<grid_for(n, 256, h->num_sms, 8), 256, 0, (cudaStream_t)stream>>>(board, score, step, max_exp, flags,
                                                                                       env_rng, n);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

// One step of b2048_rollout_many_np: b2048_step_many in rollout mode (buffer actions, ep_len bookkeeping, float32
// rewards, no auto-reset) on the generic step kernel, spawns drawn from env_rng.
int b2::launch_step_np(b2048_handle* h, const uint64_t* board_in, uint64_t* board_out, uint32_t* score, uint32_t* step,
                   uint8_t* max_exp, const uint8_t* action, const uint8_t* flags_in, const b2048_env_cfg* cfg, float* reward,
                   uint8_t* flags, int32_t* ep_len, uint32_t ep_t, int64_t n, b2048_np_rng* env_rng, cudaStream_t s) {
    StepArgs a = {};
    a.board_in = board_in; a.board_out = board_out; a.score = score; a.step = step; a.max_exp = max_exp;
    a.action = action; a.flags_in = flags_in; a.ep_len = ep_len; a.ep_t = ep_t;
    a.reward = reward; a.flags = flags; a.tables = h->d_tables; a.n = n; a.cfg = *cfg;
    if (h->smem_optin >= B2048_LUT_BYTES && n >= (int64_t)32768) {
        step_np_kernel<true, 1024><<<grid_for(n, 1024, h->num_sms, 1), 1024, B2048_LUT_BYTES, s>>>(a, env_rng);
    } else {
        step_np_kernel<false, 256><<<grid_for(n, 256, h->num_sms, 8), 256, 0, s>>>(a, env_rng);
    }
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_step_many(b2048_handle* h, const uint64_t* board_in, uint64_t* board_out, uint32_t* score,
                               uint32_t* step, uint8_t* max_exp, const uint8_t* action, uint8_t* action_out,
                               const uint8_t* flags_in, const uint8_t* spawn_replay, const b2048_env_cfg* cfg,
                               int32_t* merge_sum, float* reward,
                               double* reward64, uint8_t* flags, float* obs, int32_t* ep_len, uint32_t ep_t, int64_t n,
                               uint64_t seed, uint64_t gid0, uint32_t t, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_step_many: handle is NULL");
    B2_REQUIRE(cfg != nullptr, "b2048_step_many: cfg is NULL");
    B2_REQUIRE(n >= 0, "b2048_step_many: n < 0");
    if (n == 0) return B2048_OK;
    B2_REQUIRE(board_in && board_out && flags, "b2048_step_many: board_in/board_out/flags must not be NULL");
    B2_REQUIRE(cfg->reward_mode == B2048_REWARD_SUM || cfg->reward_mode == B2048_REWARD_LOG2,
               "b2048_step_many: unsupported reward mode");  // env.py:222-223
    B2_REQUIRE(cfg->bonus_mode >= B2048_BONUS_OFF && cfg->bonus_mode <= B2048_BONUS_LOG2,
               "b2048_step_many: unsupported bonus mode");  // env.py:248-249
    B2_REQUIRE(cfg->obs_mode >= B2048_OBS_NONE && cfg->obs_mode <= B2048_OBS_ONEHOT,
               "b2048_step_many: unsupported obs_mode");  // env.py:109-110
    B2_REQUIRE(cfg->action_mode >= B2048_ACT_BUFFER && cfg->action_mode <= B2048_ACT_PRIORITY,
               "b2048_step_many: unsupported action_mode");
    B2_REQUIRE(cfg->action_mode != B2048_ACT_BUFFER || action != nullptr,
               "b2048_step_many: action buffer required for B2048_ACT_BUFFER");
    StepArgs a;
    a.board_in = board_in; a.board_out = board_out; a.score = score; a.step = step; a.max_exp = max_exp;
    a.action = action; a.action_out = action_out; a.flags_in = flags_in; a.spawn_replay = spawn_replay; a.ep_len = ep_len; a.ep_t = ep_t;
    a.merge_sum = merge_sum;
    a.reward = reward; a.reward64 = reward64; a.flags = flags; a.obs = obs; a.tables = h->d_tables;
    a.n = n; a.seed = seed; a.gid0 = gid0; a.t = t; a.cfg = *cfg; a.keys = make_keys(seed);
    cudaStream_t s = (cudaStream_t)stream;
    a.debug_clock = debug_clock_begin(h, B2048_DBG_STEP_CLOCKS, s);
    // Large batches: persistent CTAs with the tables in shared memory.  Small batches (the B=1
    // drop-in env, unit tests): tables read through L1/L2, no 192 KB staging per launch.
    const bool use_smem = h->smem_optin >= B2048_LUT_BYTES && n >= (int64_t)32768;
    const bool all_track = score && step && max_exp, none_track = !score && !step && !max_exp;
    const bool fast = h->smem_optin >= B2048_TABLES_BYTES && n >= (int64_t)32768 && (all_track || none_track) &&
                      cfg->use_action_mask && (cfg->bonus_mode == B2048_BONUS_OFF || all_track) && reward != nullptr &&
                      reward64 == nullptr && spawn_replay == nullptr && (obs == nullptr || cfg->obs_mode == B2048_OBS_NONE) &&
                      !(h->debug & (1u << B2048_DBG_NO_FAST_STEP));
    if (fast) {
        int grid = grid_for(n, 1024, h->num_sms, 1);
        const bool pdl = !(h->debug & (1u << B2048_DBG_NO_PDL));
        cudaError_t e;
        if (cfg->action_mode == B2048_ACT_BUFFER) e = launch_fast<B2048_ACT_BUFFER>(all_track, grid, B2048_TABLES_BYTES, s, a, pdl);
        else if (cfg->action_mode == B2048_ACT_RANDOM_LEGAL) e = launch_fast<B2048_ACT_RANDOM_LEGAL>(all_track, grid, B2048_TABLES_BYTES, s, a, pdl);
        else if (cfg->action_mode == B2048_ACT_PRIORITY) e = launch_fast<B2048_ACT_PRIORITY>(all_track, grid, B2048_TABLES_BYTES, s, a, pdl);
        else e = launch_fast<B2048_ACT_RANDOM_ANY>(all_track, grid, B2048_TABLES_BYTES, s, a, pdl);
        B2_CUDA(e);
    } else if (use_smem) {
        int grid = grid_for(n, 1024, h->num_sms, 1);
        step_kernel<true, 1024><<<grid, 1024, B2048_LUT_BYTES, s>>>(a);
    } else {
        int grid = grid_for(n, 256, h->num_sms, 8);
        step_kernel<false, 256><<<grid, 256, 0, s>>>(a);
    }
    B2_CUDA(cudaGetLastError());
    if (a.debug_clock && fast) {
        long long hb[32];
        { int st = debug_clock_read(h, hb, 32, s); if (st != B2048_OK) return st; }
        for (int c = 0; c < 2; ++c) {
            long long* d = hb + 16 * c;
            fprintf(stderr, "[step clock] cta %d: start@%lld ns, staged +%lld cyc, iters:", c ? 147 : 0, d[0] - hb[0], d[2] - d[1]);
            for (int k = 3; k < 12 && d[k]; ++k) fprintf(stderr, " %lld", d[k] - d[k - 1]);
            fprintf(stderr, " | total %lld cyc, %lld ns\n", d[14] - d[1], d[15] - d[0]);
        }
    }
    return B2048_OK;
}

extern "C" int b2048_symmetries(b2048_handle* h, const uint64_t* board, const uint8_t* flags, const uint8_t* action,
                                uint64_t* board_out, uint8_t* flags_out, uint8_t* action_out, int64_t rows, int64_t n,
                                void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_symmetries: handle is NULL");
    B2_REQUIRE(rows >= 0 && n >= 0, "b2048_symmetries: negative size");
    if (rows == 0 || n == 0) return B2048_OK;
    B2_REQUIRE((board == nullptr) == (board_out == nullptr) && (flags == nullptr) == (flags_out == nullptr) &&
                   (action == nullptr) == (action_out == nullptr),
               "b2048_symmetries: every input needs its output buffer and vice versa");
    symmetries_kernel<<<grid_for(rows * n, 256, h->num_sms, 8), 256, 0, (cudaStream_t)stream>>>(
        board, flags, action, board_out, flags_out, action_out, rows, n);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_step_many_n(b2048_handle* h, uint64_t* board, uint32_t* score, uint32_t* step, uint8_t* max_exp,
                                 uint8_t* flags, int32_t flags_valid, const b2048_env_cfg* cfg, float* reward_last,
                                 float* reward_sum, int32_t* episodes, int64_t n, int32_t n_steps, uint64_t seed,
                                 uint64_t gid0, uint32_t t, void* stream) {
    B2_REQUIRE(h != nullptr && cfg != nullptr, "b2048_step_many_n: handle / cfg is NULL");
    B2_REQUIRE(n >= 0 && n_steps >= 0, "b2048_step_many_n: negative size");
    if (n == 0 || n_steps == 0) return B2048_OK;
    B2_REQUIRE(board && flags, "b2048_step_many_n: board / flags must not be NULL");
    B2_REQUIRE(cfg->action_mode == B2048_ACT_RANDOM_LEGAL || cfg->action_mode == B2048_ACT_RANDOM_ANY ||
                   cfg->action_mode == B2048_ACT_PRIORITY,
               "b2048_step_many_n: needs a device-side action mode (random_legal, random_any or priority)");
    const bool all_track = score && step && max_exp, none_track = !score && !step && !max_exp;
    const bool ok = h->smem_optin >= B2048_TABLES_BYTES && (all_track || none_track) && cfg->use_action_mask &&
                    (cfg->bonus_mode == B2048_BONUS_OFF || all_track) &&
                    (cfg->reward_mode == B2048_REWARD_SUM || cfg->reward_mode == B2048_REWARD_LOG2);
    if (!ok)
        return fail(B2048_ERR_UNSUPPORTED,
                    "b2048_step_many_n: implemented for action-mask-on configurations (the new-max-tile bonus needs the "
                    "tracked counters) with score / step / max_exp all present or all absent; call "
                    "b2048_step_many n_steps times otherwise");
    StepNArgs a;
    a.board = board; a.score = score; a.step = step; a.max_exp = max_exp; a.flags = flags; a.reward_last = reward_last;
    a.reward_sum = reward_sum; a.episodes = episodes; a.tables = h->d_tables; a.n = n; a.n_steps = n_steps;
    a.flags_valid = flags_valid; a.seed = seed; a.gid0 = gid0; a.t = t; a.cfg = *cfg; a.keys = make_keys(seed);
    const int grid = grid_for(n, 1024, h->num_sms, 1);
    cudaStream_t s = (cudaStream_t)stream;
    const bool shaped = cfg_is_shaped(*cfg);
#define B2_LAUNCH_N(A)                                                                                      \
    do {                                                                                                    \
        if (all_track && shaped) step_fast_n_kernel<A, true, true><<<grid, 1024, B2048_TABLES_BYTES, s>>>(a);    \
        else if (all_track) step_fast_n_kernel<A, true, false><<<grid, 1024, B2048_TABLES_BYTES, s>>>(a);        \
        else if (shaped) step_fast_n_kernel<A, false, true><<<grid, 1024, B2048_TABLES_BYTES, s>>>(a);           \
        else step_fast_n_kernel<A, false, false><<<grid, 1024, B2048_TABLES_BYTES, s>>>(a);                      \
    } while (0)
    if (cfg->action_mode == B2048_ACT_RANDOM_LEGAL) B2_LAUNCH_N(B2048_ACT_RANDOM_LEGAL);
    else if (cfg->action_mode == B2048_ACT_PRIORITY) B2_LAUNCH_N(B2048_ACT_PRIORITY);
    else B2_LAUNCH_N(B2048_ACT_RANDOM_ANY);
#undef B2_LAUNCH_N
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_move_many(b2048_handle* h, const uint64_t* board_in, uint64_t* board_out, const uint8_t* action,
                               int32_t* merge_sum, uint8_t* merge_info, uint8_t* flags, int64_t n, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_move_many: handle is NULL");
    B2_REQUIRE(n >= 0, "b2048_move_many: n < 0");
    if (n == 0) return B2048_OK;
    B2_REQUIRE(board_in && board_out && action, "b2048_move_many: board_in/board_out/action must not be NULL");
    move_kernel<<<grid_for(n, 256, h->num_sms, 8), 256, 0, (cudaStream_t)stream>>>(board_in, board_out, action, merge_sum,
                                                                                  merge_info, flags, h->d_tables, n);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_encode_obs(const uint64_t* board, float* obs, int32_t obs_mode, float obs_log2_scale, int64_t n,
                                void* stream) {
    B2_REQUIRE(n >= 0, "b2048_encode_obs: n < 0");
    B2_REQUIRE(obs_mode >= B2048_OBS_RAW && obs_mode <= B2048_OBS_ONEHOT, "b2048_encode_obs: unsupported obs_mode");
    if (n == 0) return B2048_OK;
    B2_REQUIRE(board && obs, "b2048_encode_obs: board/obs must not be NULL");
    int dev = 0, sms = 148;
    B2_CUDA(cudaGetDevice(&dev));
    B2_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    obs_kernel<<<grid_for(n, 256, sms, 8), 256, 0, (cudaStream_t)stream>>>(board, obs, obs_mode, obs_log2_scale, n);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}
