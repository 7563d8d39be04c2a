// The lookahead helpers of csrc/b2048_lookahead.cuh compiled with g++: the children of every board as
// lookahead_expand_kernel writes them (segments in board order here), the Q / action fold of lookahead_select_kernel, and
// step_one with a replayed spawn (b2048_step_many's body) for comparison.
#include <cstdint>
#include <vector>

#include "../../rl-2048-with-reinforce-and-actor-critic_b200/csrc/b2048_lookahead.cuh"

static std::vector<uint16_t> g_left;
static std::vector<uint8_t> g_merge;

static void ensure_lut() {
    if (!g_left.empty()) return;
    g_left.resize(65536);
    g_merge.resize(65536);
    for (uint32_t r = 0; r < 65536; ++r) {
        uint32_t o, m;
        b2::row_move_left(r, o, m);
        g_left[r] = (uint16_t)o;
        g_merge[r] = (uint8_t)m;
    }
}

extern "C" {

// Returns the number of children; boards whose segment would pass `capacity` get count 0 and first -1.
int64_t hc_lookahead_expand(const uint64_t* board, const uint8_t* flags, const uint8_t* max_exp, const b2048_env_cfg* cfg,
                            int64_t n, int64_t capacity, uint64_t* child_board, double* child_reward, uint8_t* child_done,
                            int32_t* child_first, int32_t* child_count) {
    ensure_lut();
    int64_t total = 0;
    for (int64_t i = 0; i < n; ++i) {
        const b2::Board bd = b2::make_board(board[i]);
        const uint32_t cand = b2::lookahead_candidates(*cfg, flags ? (uint32_t)flags[i] : b2::legal_mask(bd));
        b2::LookaheadMove mv[4];
        int32_t cnt[4], c = 0;
        for (int a = 0; a < 4; ++a) {
            cnt[a] = 0;
            if ((cand >> a) & 1u) {
                mv[a] = b2::lookahead_move(bd, (uint32_t)a, g_left.data(), g_merge.data(), *cfg, max_exp != nullptr);
                cnt[a] = (int32_t)b2::lookahead_children(mv[a]);
            }
            c += cnt[a];
        }
        const bool fits = total + c <= capacity;
        int64_t first = total;
        for (int a = 0; a < 4; ++a) {
            child_first[4 * i + a] = (fits && cnt[a] > 0) ? (int32_t)first : -1;
            child_count[4 * i + a] = fits ? cnt[a] : 0;
            for (int32_t j = 0; fits && j < cnt[a]; ++j) {
                b2::Board nb;
                double r;
                bool done;
                b2::lookahead_child(mv[a], (uint32_t)j, *cfg, max_exp != nullptr, max_exp ? max_exp[i] : 2u, nb, r, done);
                child_board[first + j] = b2::to_u64(nb);
                child_reward[first + j] = r;
                child_done[first + j] = (uint8_t)done;
            }
            first += cnt[a];
        }
        total += c;
    }
    return total;
}

void hc_lookahead_select(const int32_t* child_first, const int32_t* child_count, const double* child_reward,
                         const uint8_t* child_done, const float* child_value, double gamma, int64_t n, uint8_t* action,
                         double* q) {
    for (int64_t i = 0; i < n; ++i)
        action[i] = (uint8_t)b2::lookahead_select(child_first + 4 * i, child_count + 4 * i, child_reward, child_done,
                                                  child_value, gamma, q + 4 * i);
}

// step_one on (board[i], action[i]) with spawn_replay[i], auto-reset off, no step counter, max_exp (nullable) as given
void hc_step_replay(const uint64_t* board, const uint8_t* action, const uint8_t* replay, const uint8_t* max_exp,
                    const b2048_env_cfg* cfg, int64_t n, uint64_t* board_out, double* reward, uint8_t* flags) {
    ensure_lut();
    b2048_env_cfg c = *cfg;
    c.auto_reset = 0;
    c.action_mode = B2048_ACT_BUFFER;
    b2::StepOpts opt;
    opt.track_step = false;
    opt.track_max = max_exp != nullptr;
    opt.want_sum = c.reward_mode == B2048_REWARD_SUM;
    for (int64_t i = 0; i < n; ++i) {
        b2::StepIO io;
        io.board = b2::make_board(board[i]);
        io.score = 0u;
        io.step = 0u;
        io.max_exp = max_exp ? max_exp[i] : 2u;
        io.action = action[i];
        io.mask_in = 0u;
        io.have_mask_in = false;
        io.replay = replay[i];
        b2::step_one(io, c, opt, 0u, (uint64_t)i, 1u, g_left.data(), g_merge.data());
        board_out[i] = b2::to_u64(io.board);
        reward[i] = io.reward;
        flags[i] = (uint8_t)io.flags;
    }
}

}  // extern "C"
