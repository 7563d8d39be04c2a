// b2048_step.cuh — one fused environment step for one board (the body of the step kernel).
//
// Restates, in this order (reference paths relative to the reference repo):
//   Game2048.step        src/game2048.py:40-70    counters, move, score, spawn-if-changed, done
//   Game2048Env.step     src/env.py:264-302       invalid flag, reward, terminated / truncated
//   _compute_reward      src/env.py:197-261       float64, same operation order, no FMA contraction
//   get_action_mask      src/game2048.py:95-99    legal mask of the returned board
// Host+device so tests/host_check can run the identical code on the CPU against the oracle.
#pragma once
#include "../../include/b2048.h"
#include "b2048_device.cuh"
#include "b2048_np_rng.cuh"

namespace b2 {

#if defined(__CUDA_ARCH__)
B2_HD double dmul(double a, double b) { return __dmul_rn(a, b); }
B2_HD double dadd(double a, double b) { return __dadd_rn(a, b); }
#else
B2_HD double dmul(double a, double b) { volatile double r = a * b; return r; }
B2_HD double dadd(double a, double b) { volatile double r = a + b; return r; }
#endif

struct StepIO {
    // per-board state in / out
    Board board;
    uint32_t score, step, max_exp;
    // inputs
    uint32_t action;      // used when cfg.action_mode == B2048_ACT_BUFFER
    uint32_t mask_in;     // legal mask of `board` if known (have_mask_in), else recomputed when needed
    bool have_mask_in;
    uint32_t replay;      // bit 7 set: spawn replayed from the host: bits 0-3 = k-th empty cell, bit 4 = tile is a 4
    // outputs
    uint32_t action_played;
    int32_t merge_sum;
    double reward;
    uint32_t flags;
};

struct StepOpts {
    bool track_step, track_max, want_sum;
};

// kNp: the spawn is drawn from the board's NumPy env stream *np_rng (b2048_np_rng.cuh) instead of Philox, and only
// when np_draw is set.  That variant serves buffer actions without auto-reset only, so it computes no Philox block.
template <typename LutL, typename LutM, bool kNp = false>
B2_HD void step_one(StepIO& io, const b2048_env_cfg& cfg, const StepOpts& opt, uint64_t seed, uint64_t gid,
                    uint32_t t, LutL lut_left, LutM lut_merge, b2048_np_rng* np_rng = nullptr,
                    bool np_draw = false) {
    Rand4 rnd;
    if constexpr (kNp) rnd = Rand4{0u, 0u, 0u, 0u};
    else rnd = stream(seed, gid, t, B2048_DOM_STEP);

    uint32_t a;
    if (cfg.action_mode == B2048_ACT_BUFFER) {
        a = io.action & 3u;
    } else if (cfg.action_mode == B2048_ACT_RANDOM_ANY) {
        a = rnd.w2 >> 30;
    } else {
        uint32_t m = io.have_mask_in ? (io.mask_in & 0xFu) : legal_mask(io.board);
        a = cfg.action_mode == B2048_ACT_PRIORITY ? pick_priority(m, (uint32_t)cfg.action_priority) : pick_legal(m, rnd.w2);
    }
    io.action_played = a;

    if (opt.track_step) io.step += 1u;  // env.py:267 / game2048.py:47 (counts illegal moves too)

    MoveResult mv = move_board(io.board, a, lut_left, lut_merge);
    bool changed = (mv.board.lo != io.board.lo) | (mv.board.hi != io.board.hi);
    bool want_max = opt.track_max;
    MergeStats ms = merge_stats(mv.merge, opt.want_sum, want_max);
    io.merge_sum = (int32_t)ms.sum;
    io.score += ms.sum;  // game2048.py:53-54

    Board nb = mv.board;
    if (changed) {  // game2048.py:56-58
        if constexpr (kNp) {
            if (np_draw) nb = np::spawn(*np_rng, nb);
        } else if (io.replay & 0x80u) {
            nb = place_kth_empty(nb, io.replay & 0xFu, (io.replay & 0x10u) ? 2u : 1u);
        } else {
            nb = spawn(nb, rnd.w0, rnd.w1);
        }
    }
    uint32_t mask = legal_mask(nb);
    bool done = (mask == 0u) & ((nb.lo | nb.hi) != 0u);  // == _is_done() for every board incl. the empty one
    bool invalid = !changed & !done;                      // env.py:273

    double r;
    if (!cfg.use_action_mask && invalid) {
        r = cfg.invalid_action_penalty;  // env.py:206-207
    } else {
        r = (cfg.reward_mode == B2048_REWARD_SUM) ? (double)ms.sum : (double)ms.sum_log2;
        r = dmul(r, cfg.base_reward_scale);
        if (cfg.empty_tile_reward != 0.0) r = dadd(r, dmul(cfg.empty_tile_reward, (double)count_empty(nb)));
        if (cfg.merge_reward != 0.0) r = dadd(r, dmul(cfg.merge_reward, (double)ms.n));
        if (opt.track_max && ms.max_exp >= 3u && ms.max_exp > io.max_exp) {  // env.py:241
            double bonus = 0.0;
            if (cfg.bonus_mode == B2048_BONUS_RAW) bonus = (double)(1u << ms.max_exp);
            else if (cfg.bonus_mode == B2048_BONUS_LOG2) bonus = (double)ms.max_exp;
            io.max_exp = ms.max_exp;
            bonus = dmul(bonus, cfg.bonus_scale);
            r = dadd(r, bonus);
        }
        r = dadd(r, cfg.step_reward);
        if (done && cfg.endgame_penalty != 0.0) r = dadd(r, cfg.endgame_penalty);
    }
    io.reward = r;

    bool trunc = opt.track_step && cfg.max_steps > 0 && io.step >= (uint32_t)cfg.max_steps && !done;  // env.py:279-286
    uint32_t f = (changed ? B2048_F_CHANGED : 0u) | (done ? B2048_F_DONE : 0u) | (trunc ? B2048_F_TRUNC : 0u) |
                 (ms.overflow ? B2048_F_OVERFLOW : 0u);
    if (cfg.auto_reset && (done | trunc)) {
        nb = reset_board(seed, gid, t);
        io.score = 0u;
        io.step = 0u;
        io.max_exp = 2u;
        mask = legal_mask(nb);
    }
    io.board = nb;
    io.flags = f | mask;
}

// observation encode of one 16-bit row -> four float32 (env.py:131-150, raw / log2 modes)
B2_HD void encode_row(uint32_t row, int obs_mode, float scale, float out[4]) {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        uint32_t e = (row >> (4 * c)) & 0xFu;
        if (obs_mode == B2048_OBS_RAW) out[c] = e ? (float)(1u << e) : 0.0f;
        else out[c] = (float)e * scale;
    }
}

}  // namespace b2
