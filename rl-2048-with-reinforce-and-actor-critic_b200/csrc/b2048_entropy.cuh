// b2048_entropy.cuh — the entropy bonus of the policy head: the per-output term every backward kernel family adds to its head
// delta (b2048_mlp_backward_entropy).
//
// Sample s, masked logits m_j (illegal actions -1e9 like logits_to_probs, outputs j >= n_out padding), z_j = m_j - max m,
// lse = log sum_k exp z_k, p_j = exp(z_j) / sum_k exp z_k (the head's softmax):
//   H     = -sum_{legal j} p_j log p_j = lse - sum_{legal j} p_j z_j            (one logf per sample)
//   t_j   = p_j (log p_j + H) = p_j (z_j - lse + H)  for legal j < n_out, exactly 0 otherwise
// dH/dz_j = -t_j, so the ascent objective  coef log pi(a|s) + ecoef H  has the head delta
//   d_j   = coef (1[a = j] - p_j) - ecoef t_j.
// An illegal output has p_j = 0 but z_j ~ -1e9 (or -inf when padded): t_j is set to 0 by the select, never formed as 0 * inf.
// A row without a legal move has H = 0.  -1/e <= t_j <= ln 4, hence |d_j| <= |coef| + ln 4 |ecoef|: the loss scale of the
// fp16 paths comes from max(|coef| + 1.5 |ecoef|).
//
// B2_HD so that tests/host_check compiles it with g++ and compares it with a NumPy restatement.
#pragma once
#include <math.h>

#include "../../include/b2048.h"
#include "b2048_device.cuh"

namespace b2 {

// Output j's share of sum_{legal j} p_j z_j.
B2_HD float entropy_pz(float z, float p, bool legal) { return legal ? p * z : 0.0f; }

// H from lse and sum_{legal j} p_j z_j.
B2_HD float entropy_h(float lse, float sum_pz, bool any_legal) { return any_legal ? lse - sum_pz : 0.0f; }

// t_j = p_j (log p_j + H) for a legal output, 0 for an illegal or padded one.
B2_HD float entropy_term(float z, float lse, float p, float H, bool legal) { return legal ? p * ((z - lse) + H) : 0.0f; }

// A whole row held by one thread: t[0..3] and the return value H.  legal = bit j for a legal output j; bits >= n_out are ignored.
B2_HD float entropy_row(const float* z, float lse, const float* p, uint32_t legal, int n_out, float* t) {
    const uint32_t lg = legal & ((1u << n_out) - 1u);
    float spz = 0.0f;
    for (int j = 0; j < 4; ++j) spz += entropy_pz(z[j], p[j], (lg >> j) & 1u);
    const float H = entropy_h(lse, spz, lg != 0u);
    for (int j = 0; j < 4; ++j) t[j] = entropy_term(z[j], lse, p[j], H, (lg >> j) & 1u);
    return H;
}

}  // namespace b2
