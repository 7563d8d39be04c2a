/*
 * lookahead_oracle.c — TEST INFRASTRUCTURE ONLY.  The one-ply expectimax of b2048_lookahead_expand / _select restated
 * cell by cell on top of the CPU oracle (oracle/b2048_oracle.c, included here unchanged): every candidate move, every
 * spawn cell in row-major order and both tiles, the reward of _compute_reward (src/env.py:197-261) and the done test of
 * _is_done (src/game2048.py:172-187), then whole games played by the argmax of Q with a constant critic.
 *
 * Build: gcc -O2 -std=c11 -fPIC -ffp-contract=off -shared (like oracle/Makefile).
 */
#include "../../oracle/b2048_oracle.c"

/* Reward of one child, in the order of orc_step_many (the move's merges, the board after the spawn). */
static double child_reward(const b2048_env_cfg* cfg, const int merged[8], int nm, int cell[4][4], int changed, int done,
                           const uint8_t* max_exp, int seen) {
    if (!cfg->use_action_mask && !changed && !done) return cfg->invalid_action_penalty;
    double r;
    if (cfg->reward_mode == B2048_REWARD_SUM) {
        int32_t msum = 0;
        for (int k = 0; k < nm; ++k) msum += (int32_t)1 << merged[k];
        r = (double)msum;
    } else {
        r = 0.0;
        for (int k = 0; k < nm; ++k) r += (double)merged[k];
    }
    r *= cfg->base_reward_scale;
    if (cfg->empty_tile_reward != 0.0) {
        int ne = 0;
        for (int q = 0; q < 16; ++q) ne += cell[q / 4][q % 4] == 0;
        r += cfg->empty_tile_reward * (double)ne;
    }
    if (cfg->merge_reward != 0.0) r += cfg->merge_reward * (double)nm;
    int mx = 0;
    for (int k = 0; k < nm; ++k)
        if (merged[k] > mx) mx = merged[k];
    if (max_exp && mx >= 3 && mx > seen) {
        double bonus = 0.0;
        if (cfg->bonus_mode == B2048_BONUS_RAW) bonus = (double)((uint32_t)1 << mx);
        else if (cfg->bonus_mode == B2048_BONUS_LOG2) bonus = (double)mx;
        bonus *= cfg->bonus_scale;
        r += bonus;
    }
    r += cfg->step_reward;
    if (done && cfg->endgame_penalty != 0.0) r += cfg->endgame_penalty;
    return r;
}

/* Children of one board, appended at child index `base`; count[a] / first[a] per action (first = -1 without children).
 * Returns the number of children. */
static int expand_one(uint64_t b, const uint8_t* max_exp, int seen, const b2048_env_cfg* cfg, int64_t base,
                      uint64_t* child_board, double* child_reward_out, uint8_t* child_done, int32_t first[4],
                      int32_t count[4]) {
    int cell[4][4];
    unpack(b, cell);
    int cand = cfg->use_action_mask ? action_mask(cell) : 0xF;
    int c = 0;
    for (int a = 0; a < 4; ++a) {
        first[a] = -1;
        count[a] = 0;
        if (!(cand >> a & 1)) continue;
        int moved[4][4], merged[8], nm = 0, ov = 0;
        memcpy(moved, cell, sizeof(moved));
        int changed = board_move(moved, a, merged, &nm, &ov);
        first[a] = (int32_t)(base + c);
        if (!changed) {
            int done = is_done(moved);
            child_board[base + c] = pack(moved);
            child_reward_out[base + c] = child_reward(cfg, merged, nm, moved, 0, done, max_exp, seen);
            child_done[base + c] = (uint8_t)done;
            count[a] = 1;
            c += 1;
            continue;
        }
        int k = 0;
        for (int q = 0; q < 16; ++q) {
            if (moved[q / 4][q % 4] != 0) continue;
            for (int four = 0; four < 2; ++four) {
                int child[4][4];
                memcpy(child, moved, sizeof(child));
                child[q / 4][q % 4] = four ? 2 : 1;
                int done = is_done(child);
                int64_t j = base + c + 2 * k + four;
                child_board[j] = pack(child);
                child_reward_out[j] = child_reward(cfg, merged, nm, child, 1, done, max_exp, seen);
                child_done[j] = (uint8_t)done;
            }
            ++k;
        }
        count[a] = 2 * k;
        c += 2 * k;
    }
    return c;
}

int64_t orc_lookahead_expand(const uint64_t* board, const uint8_t* max_exp, const b2048_env_cfg* cfg, int64_t n,
                             uint64_t* child_board, double* child_reward_out, uint8_t* child_done, int32_t* child_first,
                             int32_t* child_count) {
    int64_t total = 0;
    for (int64_t i = 0; i < n; ++i)
        total += expand_one(board[i], max_exp ? max_exp + i : 0, max_exp ? max_exp[i] : 2, cfg, total, child_board,
                            child_reward_out, child_done, child_first + 4 * i, child_count + 4 * i);
    return total;
}

/* Whole games of boards gid0 .. gid0 + n - 1 (reset at counter 0, step t at counter t + 1, like rollout_lookahead on a
 * fresh env) played by the first argmax of Q with V(s') = v for every non-terminal child, until done / truncated or `cap`
 * steps.  Per step t < length[i]: actions / rewards (float32) / flags of step t at [t * stride + i]; final score, max_exp
 * and length per board. */
int orc_lookahead_play(uint64_t seed, uint64_t gid0, int64_t n, const b2048_env_cfg* cfg, double gamma, float v, int32_t cap,
                       int64_t stride, uint8_t* actions, float* rewards, uint8_t* flags, int32_t* length, uint32_t* score_out,
                       uint8_t* max_exp_out) {
    uint64_t cb[120];
    double cr[120];
    uint8_t cd[120];
    b2048_env_cfg c = *cfg;
    c.action_mode = B2048_ACT_BUFFER;
    c.auto_reset = 0;
    c.obs_mode = B2048_OBS_NONE;
    for (int64_t i = 0; i < n; ++i) {
        uint64_t b;
        uint32_t score = 0, step = 0;
        uint8_t mx = 2, fl = 0;
        orc_reset_many(&b, &score, &step, &mx, &fl, 0, 1, seed, gid0 + (uint64_t)i, 0);
        int32_t t = 0;
        for (; t < cap; ++t) {
            int32_t first[4], count[4];
            expand_one(b, &mx, mx, &c, 0, cb, cr, cd, first, count);
            int best = 0, any = 0;
            double best_q = 0.0;
            for (int a = 0; a < 4; ++a) {
                if (count[a] == 0) continue;
                double q;
                if (count[a] == 1) {
                    q = cr[first[a]] + gamma * (cd[first[a]] ? 0.0 : (double)v);
                } else {
                    double s = 0.0;
                    for (int k = 0; k < count[a] / 2; ++k) {
                        int j = first[a] + 2 * k;
                        double t2 = cr[j] + gamma * (cd[j] ? 0.0 : (double)v);
                        double t4 = cr[j + 1] + gamma * (cd[j + 1] ? 0.0 : (double)v);
                        s = s + (0.9 * t2 + 0.1 * t4);
                    }
                    q = s / (double)(count[a] / 2);
                }
                if (!any || q > best_q) { best = a; best_q = q; any = 1; }
            }
            uint8_t act = (uint8_t)best, f = 0;
            float r = 0.0f;
            orc_step_many(&b, &b, &score, &step, &mx, &act, 0, 0, &c, 0, &r, 0, &f, 0, 0, 1, seed, gid0 + (uint64_t)i,
                          (uint32_t)(t + 1));
            actions[t * stride + i] = act;
            rewards[t * stride + i] = r;
            flags[t * stride + i] = f;
            if (f & (B2048_F_DONE | B2048_F_TRUNC)) { ++t; break; }
        }
        length[i] = t;
        score_out[i] = score;
        max_exp_out[i] = mx;
    }
    return 0;
}
