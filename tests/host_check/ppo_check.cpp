// The PPO helpers of csrc/b2048_ppo.cuh compiled with g++: the keyed minibatch permutation, the per-slot minibatch ids as
// ppo_minibatch_kernel writes them, and the per-sample coefficients as ppo_coef_kernel computes them.
#include "../../rl-2048-with-reinforce-and-actor-critic_b200/csrc/b2048_ppo.cuh"

// out[g] = P_e(g) for every g in [0, N)
extern "C" void hc_ppo_positions(uint64_t N, uint64_t seed, uint32_t epoch, uint64_t* out) {
    for (uint64_t g = 0; g < N; ++g) out[g] = b2::ppo_position(g, N, seed, epoch);
}

// mb[t B + b] = the minibatch of global sample t n_traj + gid0 + b (ppo_minibatch_kernel)
extern "C" void hc_ppo_minibatches(int32_t T, int64_t B, int64_t n_traj, int64_t gid0, uint64_t M, uint64_t seed,
                                   uint32_t epoch, int32_t* mb) {
    const uint64_t N = (uint64_t)T * (uint64_t)n_traj;
    for (int64_t t = 0; t < T; ++t)
        for (int64_t b = 0; b < B; ++b)
            mb[t * B + b] = (int32_t)b2::ppo_minibatch((uint64_t)(t * n_traj + gid0 + b), N, M, seed, epoch);
}

// per sample i: out[8 i ..] = {logp, ratio, coef, gcoef, clipped, kl, surrogate, value_loss}
extern "C" void hc_ppo_samples(const float* logits, const uint8_t* legal, const uint8_t* action, const double* logp_old,
                               const float* adv, const float* ret, const float* v_old, const float* v, int64_t n,
                               double mb_size, double clip_eps, double vclip_eps, int32_t huber, double huber_delta,
                               double* out) {
    for (int64_t i = 0; i < n; ++i) {
        const b2::PpoSample p = b2::ppo_sample(logits + 4 * i, legal[i], action[i], logp_old[i], adv[i], ret[i], v_old[i], v[i],
                                               mb_size, clip_eps, vclip_eps, huber, huber_delta);
        const double row[8] = {p.logp, p.ratio, p.coef, p.gcoef, p.clipped, p.kl, p.surrogate, p.value_loss};
        for (int k = 0; k < 8; ++k) out[8 * i + k] = row[k];
    }
}
