// The per-lane recurrence of the fixed-horizon window targets (csrc/b2048_horizon.cuh), compiled with g++ for a bit-exact
// comparison with a NumPy float64 restatement.  The wrapper forms c and 1 / (T n_traj) as b2048_segment_targets does.
#include "../../rl-2048-with-reinforce-and-actor-critic_b200/csrc/b2048_horizon.cuh"

extern "C" void hc_segment_targets(const float* reward, const uint8_t* flags, const float* value, int32_t T, int64_t B,
                                   double gamma, double lambda, int32_t huber, float huber_delta, float n_traj, float* v,
                                   float* td, float* gcoef, int32_t* valid_len) {
    const double c = value ? gamma * lambda : gamma;
    const float inv_div = 1.0f / ((float)T * n_traj);
    for (int64_t b = 0; b < B; ++b)
        valid_len[b] = b2::segment_lane(reward + b, flags + b, value ? value + b : nullptr, B, T, (float)gamma, c, huber,
                                        huber_delta, inv_div, v + b, td ? td + b : nullptr, gcoef ? gcoef + b : nullptr);
}
