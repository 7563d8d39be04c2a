// b2048_horizon.cuh — per-lane targets of a fixed-horizon window with reset-on-done (several episodes per lane).
//
// A window is T steps of B lanes played with auto-reset; e_t = (flags[t+1] & (DONE | TRUNC)) != 0 marks the last step
// of an episode (boards[t+1] is then the reset board).  Returns, TD errors and advantages restart at every e_t; a
// truncated episode is not bootstrapped, exactly like update_batch's last step (td_error_kernel's [t+1 < len]).
//
//   REINFORCE      G_t = r_t + gamma (1 - e_t) G_{t+1}; only slots whose episode ends inside the window are samples:
//                  valid_len = (last boundary) + 1, or 0; v = 0 on the unused tail.
//   actor-critic   delta_t = r_t + gamma (1 - e_t) V(s_{t+1}) - V(s_t) (V(boards[T]) bootstraps the cut-off tail),
//                  A_t = delta_t + gamma lambda (1 - e_t) A_{t+1}; every slot is a sample (valid_len = T);
//                  gcoef = dLoss/dV of delta (mse or Huber, _get_grad_logits_critic) / (T n_traj).
//
// B2_HD so that tests/host_check compiles the recurrence with g++ (-ffp-contract=off) and compares it bit for bit with a
// NumPy float64 restatement: the float32 TD arithmetic uses separately rounded operations (no FMA contraction) on both
// sides, the recurrence runs in float64 like reverse_scan_kernel.
//
// Bootstrapping at truncation (opt-in, ReinforceAgent.update_from_horizon / update_from_rollout(bootstrap_truncation=True)):
// a TRUNC boundary ends an episode only because the step budget ran out, so its target is r + gamma V(s') with s' the
// board the episode was cut on.  fold_bootstrap folds gamma V(s') into a copy of the rewards; segment_lane (vn = 0 at a
// boundary: r' + gamma 0 == r' exactly) then computes every target, TD error, GAE term and gcoef bit for bit as with
// vn = V(s') at that boundary.  s' is gone from a reset-on-done window (boards[t + 1] is the reset board), but spawns are
// counter-based: pre_reset_board replays it from (boards[t], actions[t], seed, gid, t_env) with step_one itself.
#pragma once
#include "../../include/b2048.h"
#include "b2048_device.cuh"
#include "b2048_step.cuh"

namespace b2 {

B2_HD float f32_mul(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fmul_rn(a, b);
#else
    return a * b;
#endif
}
B2_HD float f32_add(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fadd_rn(a, b);
#else
    return a + b;
#endif
}
B2_HD double f64_mul(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}
B2_HD double f64_add(double a, double b) {
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

// One lane of the window, element t at index t * stride.  rewards [T], flags [T + 1], value [T + 1] or NULL (REINFORCE).
// c = gamma (REINFORCE) or gamma * lambda (actor-critic); inv_div = 1 / (T n_traj).  Writes v [T] (returns-to-go or
// advantages) and, with a value, td / gcoef [T]; returns valid_len.
B2_HD int segment_lane(const float* reward, const uint8_t* flags, const float* value, int64_t stride, int T, float gamma,
                       double c, int huber, float huber_delta, float inv_div, float* v, float* td, float* gcoef) {
    int valid = value ? T : 0;
    double G = 0.0;
    for (int t = T - 1; t >= 0; --t) {
        const int64_t i = (int64_t)t * stride;
        const bool e = (flags[i + stride] & (B2048_F_DONE | B2048_F_TRUNC)) != 0;
        if (e && valid == 0) valid = t + 1;
        float x = reward[i];
        if (value) {
            const float vc = value[i];
            const float vn = e ? 0.0f : value[i + stride];
            const float target = f32_add(x, f32_mul(gamma, vn));
            const float diff = f32_add(vc, -target);     // dLoss/dV of the mse loss
            float g = diff;
            if (huber && (diff > huber_delta || diff < -huber_delta)) g = diff > 0.0f ? huber_delta : -huber_delta;
            x = f32_add(target, -vc);                    // delta
            td[i] = x;
            gcoef[i] = f32_mul(g, inv_div);
        }
        G = e ? (double)x : f64_add((double)x, f64_mul(c, G));
        v[i] = (value || t < valid) ? (float)G : 0.0f;
    }
    return valid;
}

// The bootstrapped reward of a truncated episode's last step: r + gamma V(s'), each operation rounded separately.
B2_HD float fold_bootstrap(float r, float gamma, float v_next) { return f32_add(r, f32_mul(gamma, v_next)); }

// The board after `a` on `board` at env counter t_env of lane gid, before an auto-reset replaced it: the move, then the
// Philox spawn of (seed, gid, t_env) when the move changed the board.  step_one with auto-reset off computes exactly that;
// counters, rewards and flags are not needed.
template <typename LutL, typename LutM>
B2_HD uint64_t pre_reset_board(uint64_t board, uint32_t a, uint64_t seed, uint64_t gid, uint32_t t_env, LutL lut_left,
                               LutM lut_merge) {
    b2048_env_cfg cfg = {};
    cfg.action_mode = B2048_ACT_BUFFER;
    cfg.use_action_mask = 1;
    StepIO io = {};
    io.board = make_board(board);
    io.max_exp = 2u;
    io.action = a;
    const StepOpts opt = {false, false, false};
    step_one(io, cfg, opt, seed, gid, t_env, lut_left, lut_merge);
    return to_u64(io.board);
}

// The largest tile of an episode that ended with the move `a` on `board` (max_tile_seen): every tile >= 8 came from a
// merge, so it is the largest tile after that move (a 15+15 merge counts as exponent 16), and at least 4.
template <typename LutL, typename LutM>
B2_HD uint32_t final_max_exp(uint64_t board, uint32_t a, LutL lut_left, LutM lut_merge) {
    const MoveResult r = move_board(make_board(board), a & 3u, lut_left, lut_merge);
    uint32_t m = merge_stats(r.merge, false, true).max_exp;
    const uint64_t b = to_u64(r.board);
    for (int k = 0; k < 16; ++k) {
        const uint32_t e = (uint32_t)((b >> (4 * k)) & 0xFull);
        m = e > m ? e : m;
    }
    return m > 2u ? m : 2u;
}

}  // namespace b2
