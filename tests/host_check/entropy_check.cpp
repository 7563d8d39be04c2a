// The entropy helper of csrc/b2048_entropy.cuh compiled with g++: the head's masked softmax as the backward kernels form it
// (illegal logits -1e9, outputs j >= n_out -inf), then H and t_j = p_j (log p_j + H) of every row.
#include <math.h>

#include "../../rl-2048-with-reinforce-and-actor-critic_b200/csrc/b2048_entropy.cuh"

// per row i: p[4 i ..], t[4 i ..], H[i]; legal[i] = the row's mask bits (use_mask = 0: every output below n_out is legal)
extern "C" void hc_entropy_rows(const float* logits, const uint8_t* legal, int32_t use_mask, int32_t n_out, int64_t n, float* p,
                                float* t, float* H) {
    for (int64_t i = 0; i < n; ++i) {
        const uint32_t fl = use_mask ? legal[i] : 0xFu;
        float m[4], z[4], e[4], q[4], sum = 0.0f;
        for (int j = 0; j < 4; ++j) m[j] = j >= n_out ? -INFINITY : ((use_mask && !((fl >> j) & 1u)) ? -1e9f : logits[4 * i + j]);
        const float mx = fmaxf(fmaxf(m[0], m[1]), fmaxf(m[2], m[3]));
        for (int j = 0; j < 4; ++j) { z[j] = m[j] - mx; e[j] = expf(z[j]); sum += e[j]; }
        for (int j = 0; j < 4; ++j) q[j] = e[j] / sum;
        H[i] = b2::entropy_row(z, logf(sum), q, fl, n_out, t + 4 * i);
        for (int j = 0; j < 4; ++j) p[4 * i + j] = q[j];
    }
}
