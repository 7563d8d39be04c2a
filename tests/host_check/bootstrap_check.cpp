// The bootstrapping helpers of csrc/b2048_horizon.cuh compiled with g++: the pre-reset replay of a truncated episode's last
// board (step_one with auto-reset off) and the fold of gamma V(s') into the rewards, as the kernels apply them per slot.
#include <vector>

#include "../../rl-2048-with-reinforce-and-actor-critic_b200/csrc/b2048_horizon.cuh"

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

// one board per element, each with its own seed, global id and env counter
extern "C" void hc_pre_reset_many(const uint64_t* board, const uint8_t* action, const uint64_t* seed, const uint64_t* gid,
                                  const uint32_t* t_env, uint64_t* out, int64_t n) {
    ensure_lut();
    for (int64_t i = 0; i < n; ++i)
        out[i] = b2::pre_reset_board(board[i], action[i], seed[i], gid[i], t_env[i], g_left.data(), g_merge.data());
}

// b2048_fold_bootstrap's result: a copy of reward[n] with reward + gamma value[k] at slots[k]
extern "C" void hc_fold_bootstrap(const float* reward, const int64_t* slots, const float* value, int64_t K, int64_t n,
                                  float gamma, float* out) {
    for (int64_t i = 0; i < n; ++i) out[i] = reward[i];
    for (int64_t k = 0; k < K; ++k) out[slots[k]] = b2::fold_bootstrap(reward[slots[k]], gamma, value[k]);
}
