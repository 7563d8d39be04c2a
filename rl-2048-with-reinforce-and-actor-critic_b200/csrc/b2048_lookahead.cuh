// b2048_lookahead.cuh — the one-ply expectimax over a learned critic (DESIGN.md K7): the children of every candidate move
// of a board, and the fold of their values into Q(s, a) and an action.
//
// Host+device so tests/host_check can run the identical code on the CPU against the cell-by-cell oracle enumeration.
//   children of a move  Game2048.step with every spawn (game2048.py:40-70, :108-118) + _compute_reward (env.py:197-261),
//                       restated from step_one (b2048_step.cuh) with auto-reset and truncation off: the child of (k, v) is
//                       bit-identical to b2048_step_many with spawn_replay = 0x80 | k | (v == 4) << 4
//   Q / action          sum over the spawns of p (r + gamma V(s')) with the rules' probabilities 1/n, 0.9 and 0.1; first
//                       argmax over the candidates (the greedy tie rule, reinforce_agent.py:179-185)
#pragma once
#include "b2048_step.cuh"

namespace b2 {

constexpr int LOOKAHEAD_MAX_CHILDREN = 120;   // 4 moves x 15 empty cells x {2, 4}

#if defined(__CUDA_ARCH__)
B2_HD double ddiv(double a, double b) { return __ddiv_rn(a, b); }
B2_HD double qnan() { return __longlong_as_double(0x7FF8000000000000ll); }
#else
B2_HD double ddiv(double a, double b) { volatile double r = a / b; return r; }
B2_HD double qnan() { return __builtin_nan(""); }
#endif

// One move of a board, before the spawn: everything its children share.
struct LookaheadMove {
    Board moved;       // board after the move, before any spawn
    bool changed;
    uint32_t n_empty;  // empty cells of `moved`
    MergeStats ms;
};

template <typename LutL, typename LutM>
B2_HD LookaheadMove lookahead_move(Board b, uint32_t a, LutL lut_left, LutM lut_merge, const b2048_env_cfg& cfg,
                                   bool track_max) {
    LookaheadMove m;
    MoveResult mv = move_board(b, a, lut_left, lut_merge);
    m.moved = mv.board;
    m.changed = (mv.board.lo != b.lo) | (mv.board.hi != b.hi);
    m.n_empty = (uint32_t)count_empty(mv.board);
    m.ms = merge_stats(mv.merge, cfg.reward_mode == B2048_REWARD_SUM, track_max);
    return m;
}

// Children of a candidate move: 2 n for a changed move with n empty cells, 1 (the unchanged board) otherwise.
B2_HD uint32_t lookahead_children(const LookaheadMove& m) { return m.changed ? 2u * m.n_empty : 1u; }

// Child j of a move (j = 2 k + (tile is a 4) for a changed move, j = 0 for an unchanged one): the board, float64 reward
// and done flag of step_one on the same board and action with that spawn replayed, auto-reset off, no step counter and
// the new-max-tile bonus against max_exp (track_max = max_exp was given).
B2_HD void lookahead_child(const LookaheadMove& m, uint32_t j, const b2048_env_cfg& cfg, bool track_max, uint32_t max_exp,
                           Board& nb, double& r, bool& done) {
    nb = m.moved;
    if (m.changed) nb = place_kth_empty(nb, j >> 1, (j & 1u) ? 2u : 1u);
    done = (legal_mask(nb) == 0u) & ((nb.lo | nb.hi) != 0u);
    const bool invalid = !m.changed & !done;
    if (!cfg.use_action_mask && invalid) {
        r = cfg.invalid_action_penalty;
        return;
    }
    r = (cfg.reward_mode == B2048_REWARD_SUM) ? (double)m.ms.sum : (double)m.ms.sum_log2;
    r = dmul(r, cfg.base_reward_scale);
    if (cfg.empty_tile_reward != 0.0) r = dadd(r, dmul(cfg.empty_tile_reward, (double)count_empty(nb)));
    if (cfg.merge_reward != 0.0) r = dadd(r, dmul(cfg.merge_reward, (double)m.ms.n));
    if (track_max && m.ms.max_exp >= 3u && m.ms.max_exp > max_exp) {
        double bonus = 0.0;
        if (cfg.bonus_mode == B2048_BONUS_RAW) bonus = (double)(1u << m.ms.max_exp);
        else if (cfg.bonus_mode == B2048_BONUS_LOG2) bonus = (double)m.ms.max_exp;
        r = dadd(r, dmul(bonus, cfg.bonus_scale));
    }
    r = dadd(r, cfg.step_reward);
    if (done && cfg.endgame_penalty != 0.0) r = dadd(r, cfg.endgame_penalty);
}

// The candidate moves of a board: its legal mask with the action mask on, all four actions with it off.
B2_HD uint32_t lookahead_candidates(const b2048_env_cfg& cfg, uint32_t legal) {
    return cfg.use_action_mask ? (legal & 0xFu) : 0xFu;
}

// t = r + gamma V(s'), V(s') = 0 for a terminal child; V is the float32 critic output widened to float64.
B2_HD double lookahead_target(double r, bool done, float v, double gamma) {
    return dadd(r, dmul(gamma, done ? 0.0 : (double)v));
}

// Q of one candidate move from its `count` children starting at child index `first`:
//   count == 1 (unchanged move): Q = t;
//   count == 2 n: S = sum over k = 0 .. n-1, in order, of (0.9 t(k, 2) + 0.1 t(k, 4)), Q = S / n.
template <typename Rw, typename Dn, typename Vl>
B2_HD double lookahead_q(int64_t first, int32_t count, Rw reward, Dn done, Vl value, double gamma) {
    if (count == 1) return lookahead_target(reward[first], done[first] != 0, value[first], gamma);
    double s = 0.0;
    for (int32_t k = 0; k < count / 2; ++k) {
        const int64_t c = first + 2 * k;
        const double t2 = lookahead_target(reward[c], done[c] != 0, value[c], gamma);
        const double t4 = lookahead_target(reward[c + 1], done[c + 1] != 0, value[c + 1], gamma);
        s = dadd(s, dadd(dmul(0.9, t2), dmul(0.1, t4)));
    }
    return ddiv(s, (double)(count / 2));
}

// The action of a board: the first candidate (count > 0) with the largest Q under `>`; 0 when there is none.  q[a] is
// NaN for a non-candidate.
template <typename Rw, typename Dn, typename Vl>
B2_HD uint32_t lookahead_select(const int32_t first[4], const int32_t count[4], Rw reward, Dn done, Vl value, double gamma,
                                double q[4]) {
    uint32_t best = 0u;
    bool any = false;
    double best_q = 0.0;
    for (uint32_t a = 0; a < 4u; ++a) {
        if (count[a] <= 0) {
            q[a] = qnan();
            continue;
        }
        q[a] = lookahead_q(first[a], count[a], reward, done, value, gamma);
        if (!any || q[a] > best_q) {
            best = a;
            best_q = q[a];
            any = true;
        }
    }
    return best;
}

}  // namespace b2
