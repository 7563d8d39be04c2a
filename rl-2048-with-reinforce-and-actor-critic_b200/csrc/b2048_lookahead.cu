// b2048_lookahead.cu — one-ply expectimax over a learned critic (DESIGN.md K7) and its C entry points.
//
//   lookahead_expand_kernel  one thread per listed board: every candidate move once, then all its (cell, tile) spawns,
//                            written to one compacted child array (board u64, reward f64, done u8); each board's segment
//                            is reserved with one atomic per warp, and its contents do not depend on where it lands
//   lookahead_select_kernel  one thread per listed board: folds r + gamma V(s') of its children into Q(s, a) (float64) and
//                            the first argmax over the candidates
//
// Between the two the caller evaluates the critic on the children (b2048_mlp_forward on child_board[0 .. total)).
#include <cuda_runtime.h>

#include "b2048_internal.h"
#include "b2048_lookahead.cuh"

namespace b2 {

struct ExpandArgs {
    const uint64_t* board;
    const uint8_t* flags;      // nullable: legal masks recomputed
    const uint8_t* max_exp;    // nullable: no new-max-tile bonus
    const int32_t* slot_map;   // nullable: boards 0 .. n - 1
    const int32_t* n_dev;      // nullable: the number of listed boards is min(n_slots, *n_dev)
    int64_t n_slots;
    int64_t capacity;
    uint64_t* child_board;
    double* child_reward;
    uint8_t* child_done;
    int32_t* child_first;      // [B, 4]
    int32_t* child_count;      // [B, 4]
    int32_t* total;
    const uint8_t* tables;
    b2048_env_cfg cfg;
};

__global__ void __launch_bounds__(256) lookahead_expand_kernel(const __grid_constant__ ExpandArgs args) {
    const int64_t n = args.n_dev ? min(args.n_slots, (int64_t)*args.n_dev) : args.n_slots;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = i < n;
    const int lane = threadIdx.x & 31;
    const uint16_t* lut_left = reinterpret_cast<const uint16_t*>(args.tables);
    const uint8_t* lut_merge = args.tables + B2048_LUT_LEFT_BYTES;
    const b2048_env_cfg& cfg = args.cfg;
    const bool track_max = args.max_exp != nullptr;

    int64_t b = 0;
    Board bd{0u, 0u};
    uint32_t cand = 0u, mx = 2u;
    if (valid) {
        b = args.slot_map ? (int64_t)args.slot_map[i] : i;
        bd = make_board(args.board[b]);
        const uint32_t legal = args.flags ? (uint32_t)args.flags[b] : legal_mask(bd);
        cand = lookahead_candidates(cfg, legal);
        if (track_max) mx = args.max_exp[b];
    }
    LookaheadMove mv[4];
    int32_t cnt[4];
    int32_t c = 0;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        cnt[a] = 0;
        if ((cand >> a) & 1u) {
            mv[a] = lookahead_move(bd, (uint32_t)a, lut_left, lut_merge, cfg, track_max);
            cnt[a] = (int32_t)lookahead_children(mv[a]);
        }
        c += cnt[a];
    }
    // warp-aggregated reservation: inclusive scan of the counts, one atomic per warp
    int32_t incl = c;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int32_t o = __shfl_up_sync(0xFFFFFFFFu, incl, d);
        if (lane >= d) incl += o;
    }
    int32_t base = 0;
    if (lane == 31 && incl > 0) base = atomicAdd(args.total, incl);
    base = __shfl_sync(0xFFFFFFFFu, base, 31) + incl - c;
    if (!valid) return;
    const bool fits = (int64_t)base + c <= args.capacity;
    int32_t first = base;
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        args.child_first[4 * b + a] = (fits && cnt[a] > 0) ? first : -1;
        args.child_count[4 * b + a] = fits ? cnt[a] : 0;
        if (fits) {
            for (int32_t j = 0; j < cnt[a]; ++j) {
                Board nb;
                double r;
                bool done;
                lookahead_child(mv[a], (uint32_t)j, cfg, track_max, mx, nb, r, done);
                args.child_board[first + j] = to_u64(nb);
                args.child_reward[first + j] = r;
                args.child_done[first + j] = (uint8_t)done;
            }
        }
        first += cnt[a];
    }
}

__global__ void __launch_bounds__(256) lookahead_select_kernel(const int32_t* __restrict__ slot_map,
                                                                const int32_t* __restrict__ n_dev, int64_t n_slots,
                                                                const int32_t* __restrict__ child_first,
                                                                const int32_t* __restrict__ child_count,
                                                                const double* __restrict__ child_reward,
                                                                const uint8_t* __restrict__ child_done,
                                                                const float* __restrict__ child_value, double gamma,
                                                                uint8_t* __restrict__ action, double* __restrict__ q) {
    const int64_t n = n_dev ? min(n_slots, (int64_t)*n_dev) : n_slots;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const int64_t b = slot_map ? (int64_t)slot_map[i] : i;
    const int4 f4 = reinterpret_cast<const int4*>(child_first)[b];
    const int4 c4 = reinterpret_cast<const int4*>(child_count)[b];
    const int32_t first[4] = {f4.x, f4.y, f4.z, f4.w}, count[4] = {c4.x, c4.y, c4.z, c4.w};
    double qa[4];
    action[b] = (uint8_t)lookahead_select(first, count, child_reward, child_done, child_value, gamma, qa);
    if (q) {
#pragma unroll
        for (int a = 0; a < 4; ++a) q[4 * b + a] = qa[a];
    }
}

}  // namespace b2

// ================================================================================================ C ABI
using namespace b2;

extern "C" int b2048_lookahead_expand(b2048_handle* h, const uint64_t* board, const uint8_t* flags, const uint8_t* max_exp,
                                      const b2048_env_cfg* cfg, const int32_t* slot_map, int64_t n_slots,
                                      const int32_t* n_slots_dev, int64_t B, int64_t capacity, uint64_t* child_board,
                                      double* child_reward, uint8_t* child_done, int32_t* child_first, int32_t* child_count,
                                      int32_t* total_dev, void* stream) {
    B2_REQUIRE(h != nullptr && cfg != nullptr, "b2048_lookahead_expand: handle / cfg is NULL");
    B2_REQUIRE(B >= 0 && n_slots >= 0 && n_slots <= B, "b2048_lookahead_expand: n_slots out of [0, B]");
    B2_REQUIRE(n_slots <= (int64_t)INT32_MAX / LOOKAHEAD_MAX_CHILDREN && capacity >= 0 && capacity <= (int64_t)INT32_MAX,
               "b2048_lookahead_expand: n_slots * 120 and capacity must fit in int32");
    B2_REQUIRE(slot_map != nullptr || n_slots_dev == nullptr, "b2048_lookahead_expand: n_slots_dev needs a slot_map");
    B2_REQUIRE(total_dev != nullptr, "b2048_lookahead_expand: total_dev is NULL");
    B2_REQUIRE(cfg->reward_mode == B2048_REWARD_SUM || cfg->reward_mode == B2048_REWARD_LOG2,
               "b2048_lookahead_expand: unsupported reward mode");
    B2_REQUIRE(cfg->bonus_mode >= B2048_BONUS_OFF && cfg->bonus_mode <= B2048_BONUS_LOG2,
               "b2048_lookahead_expand: unsupported bonus mode");
    cudaStream_t s = (cudaStream_t)stream;
    B2_CUDA(cudaMemsetAsync(total_dev, 0, sizeof(int32_t), s));
    if (n_slots == 0) return B2048_OK;
    B2_REQUIRE(board && child_first && child_count && (capacity == 0 || (child_board && child_reward && child_done)),
               "b2048_lookahead_expand: NULL buffer");
    ExpandArgs a;
    a.board = board; a.flags = flags; a.max_exp = max_exp; a.slot_map = slot_map; a.n_dev = n_slots_dev;
    a.n_slots = n_slots; a.capacity = capacity; a.child_board = child_board; a.child_reward = child_reward;
    a.child_done = child_done; a.child_first = child_first; a.child_count = child_count; a.total = total_dev;
    a.tables = h->d_tables; a.cfg = *cfg;
    lookahead_expand_kernel<<<(unsigned)((n_slots + 255) / 256), 256, 0, s>>>(a);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_lookahead_select(b2048_handle* h, const int32_t* slot_map, int64_t n_slots, const int32_t* n_slots_dev,
                                      int64_t B, const int32_t* child_first, const int32_t* child_count,
                                      const double* child_reward, const uint8_t* child_done, const float* child_value,
                                      double gamma, uint8_t* action, double* q, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_lookahead_select: handle is NULL");
    B2_REQUIRE(B >= 0 && n_slots >= 0 && n_slots <= B, "b2048_lookahead_select: n_slots out of [0, B]");
    B2_REQUIRE(slot_map != nullptr || n_slots_dev == nullptr, "b2048_lookahead_select: n_slots_dev needs a slot_map");
    if (n_slots == 0) return B2048_OK;
    B2_REQUIRE(child_first && child_count && action, "b2048_lookahead_select: NULL buffer");
    lookahead_select_kernel<<<(unsigned)((n_slots + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        slot_map, n_slots_dev, n_slots, child_first, child_count, child_reward, child_done, child_value, gamma, action, q);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}
