// b2048_ppo.cuh — PPO on fixed-horizon windows: the world-size-invariant minibatch partition and the per-sample
// clipped-surrogate / clipped-value coefficients fed to b2048_mlp_backward.
//
// Partition.  Slot (t, b) of a window has the global sample index g = t n_traj + gid0 + b in [0, N), N = T n_traj
// (n_traj = the global lane count, gid0 = the global id of the shard's lane 0).  Epoch e permutes [0, N) with a keyed
// bijection P_e: a 4-round balanced Feistel network on 2h bits, h = max(1, ceil(ceil(log2 N) / 2)); round r maps
// (L, R) -> (R, L ^ F_r(R)) with F_r(R) = philox4x32_10(counter (R, r, e, B2048_DOM_PPO), key shuffle_seed).w0 masked to
// h bits; values >= N are walked through the network again until they land in [0, N).  Minibatch of g:
// m = floor(P_e(g) M / N), so minibatch m holds ceil((m + 1) N / M) - ceil(m N / M) samples wherever they live: every
// rank knows the global sizes without a message, and the all-reduced gradient is the single-process one.
//
// Coefficients (one sample s of minibatch m, |mb| its global size; float64 from float32 network outputs):
//   logp  = masked log-softmax of the logits at a_s (illegal actions filled with -1e9 like logits_to_probs)
//   r     = exp(logp - logp_old)
//   coef  = A r / |mb|, 0 when (A > 0 and r > 1 + eps) or (A < 0 and r < 1 - eps): d/dlogp of mean min(r A, clip(r) A)
//   d     = V - R; with value clipping V_c = V_old + clamp(V - V_old, -eps_v, eps_v) and the larger of (V - R)^2,
//           (V_c - R)^2 selects the gradient (V - R), or (V_c - R) [|V - V_old| < eps_v]; Huber clips the selected one
//   gcoef = that dLoss/dV / |mb|  (critic descent, like segment_lane's gcoef)
//
// B2_HD so that tests/host_check compiles it with g++ and compares it with NumPy restatements.
#pragma once
#include <math.h>

#include "../../include/b2048.h"
#include "b2048_device.cuh"

namespace b2 {

// h of the Feistel network on [0, N): half of ceil(log2 N) bits, rounded up, at least 1.
B2_HD int ppo_half_bits(uint64_t N) {
    int bits = 0;
    while (bits < 64 && (1ull << bits) < N) ++bits;
    const int h = (bits + 1) / 2;
    return h < 1 ? 1 : h;
}

// P_e(g): the position of global sample g in epoch `epoch`'s permutation of [0, N).  g < N <= 2^32.
B2_HD uint64_t ppo_position(uint64_t g, uint64_t N, uint64_t seed, uint32_t epoch) {
    const int h = ppo_half_bits(N);
    const uint64_t mask = (1ull << h) - 1ull;
    const uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
    uint64_t x = g;
    do {
        uint64_t L = x >> h, R = x & mask;
        for (uint32_t r = 0; r < 4; ++r) {
            const uint64_t F = philox4x32_10((uint32_t)R, r, epoch, B2048_DOM_PPO, k0, k1).w0 & mask;
            const uint64_t nl = R;
            R = L ^ F;
            L = nl;
        }
        x = (L << h) | R;
    } while (x >= N);
    return x;
}

// The minibatch of global sample g: floor(P_e(g) M / N), M <= N <= 2^32.
B2_HD uint32_t ppo_minibatch(uint64_t g, uint64_t N, uint64_t M, uint64_t seed, uint32_t epoch) {
    return (uint32_t)(ppo_position(g, N, seed, epoch) * M / N);
}

// log pi(a | s) from one sample's four float32 logits, in float64; legal = the 4-bit legal mask (0xF: no masking).
B2_HD double ppo_logp(const float* z, uint32_t legal, uint32_t a) {
    double x[4], mx = -INFINITY, xa = 0.0;
    for (int i = 0; i < 4; ++i) {
        x[i] = ((legal >> i) & 1u) ? (double)z[i] : -1e9;
        mx = x[i] > mx ? x[i] : mx;
        xa = (uint32_t)i == (a & 3u) ? x[i] : xa;      // no dynamic index: x stays in registers
    }
    double s = 0.0;
    for (int i = 0; i < 4; ++i) s += exp(x[i] - mx);
    return (xa - mx) - log(s);
}

struct PpoSample {
    double logp, ratio, coef, gcoef;
    double clipped;     // 1 when the actor coefficient was clipped to 0
    double kl;          // r - 1 - log r (approximate KL(old || new))
    double surrogate;   // min(r A, clip(r, 1 - eps, 1 + eps) A)
    double value_loss;  // 0.5 e^2 (mse) or the Huber loss of the selected value error e
};

// One sample's coefficients (see the top of the file).  vclip_eps <= 0: no value clipping.
B2_HD PpoSample ppo_sample(const float* z, uint32_t legal, uint32_t a, double logp_old, float adv, float ret, float v_old,
                           float v, double mb_size, double clip_eps, double vclip_eps, int huber, double huber_delta) {
    PpoSample p;
    p.logp = ppo_logp(z, legal, a);
    p.ratio = exp(p.logp - logp_old);
    const double A = (double)adv, r = p.ratio;
    const bool clip = (A > 0.0 && r > 1.0 + clip_eps) || (A < 0.0 && r < 1.0 - clip_eps);
    p.clipped = clip ? 1.0 : 0.0;
    p.coef = clip ? 0.0 : A * r / mb_size;
    const double rc = r < 1.0 - clip_eps ? 1.0 - clip_eps : (r > 1.0 + clip_eps ? 1.0 + clip_eps : r);
    p.surrogate = r * A < rc * A ? r * A : rc * A;
    p.kl = (r - 1.0) - (p.logp - logp_old);
    const double R = (double)ret, V = (double)v, d = V - R;
    double e = d, g = d;
    if (vclip_eps > 0.0) {
        const double dv = V - (double)v_old;
        const double vc = (double)v_old + (dv < -vclip_eps ? -vclip_eps : (dv > vclip_eps ? vclip_eps : dv));
        const double dc = vc - R;
        if (dc * dc > d * d) {
            e = dc;
            g = (dv < vclip_eps && dv > -vclip_eps) ? dc : 0.0;
        }
    }
    const double ae = e < 0.0 ? -e : e;
    if (huber) {
        if (g > huber_delta) g = huber_delta;
        if (g < -huber_delta) g = -huber_delta;
        p.value_loss = ae <= huber_delta ? 0.5 * e * e : huber_delta * (ae - 0.5 * huber_delta);
    } else {
        p.value_loss = 0.5 * e * e;
    }
    p.gcoef = g / mb_size;
    return p;
}

}  // namespace b2
