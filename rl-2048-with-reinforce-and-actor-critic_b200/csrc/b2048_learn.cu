// b2048_learn.cu — returns / advantages / policy-gradient update kernels (fp32 CUDA-core path).
//
//   K4 reverse_scan_kernel       compute_returns            src/reinforce_agent.py:255-273
//      reverse_scan_warp_kernel  same, warp-shuffle affine suffix scan over time for small batches
//   K5 weighted_stats_kernel     _compute_weighted_stats    src/reinforce_agent.py:864-881
//      advantage_kernel          _compute_advantages        src/reinforce_agent.py:276-325 (+ the 1/(T n) weight, :533-534)
//      td_error_kernel           TD(0) targets / errors     src/reinforce_agent.py:439-447, :884-910
//      segment_targets_kernel    returns / TD / GAE of fixed-horizon windows (episode boundaries inside a lane)
//      advantage_window_kernel   advantage_kernel with the window's T n_traj divisor
//      horizon_episodes_kernel   episodes completed inside a window (logging)
//      replay_pre_reset_kernel   the boards truncated episodes were cut on (bootstrapping at truncation)
//      fold_bootstrap_kernel     r + gamma V(s') at the truncated slots of a copy of the rewards
//   K6 mlp_backward_kernel       _backpropagation per tile  src/reinforce_agent.py:639-678 (deltas + activations)
//      atb_kernel                dW_l = A_l^T D_l           (sum over samples of np.outer, :666)
//      colsum_kernel             db_l = sum_s D_l
//      sumsq / clip / sgd / adam clip_grads_global_norm :835-861, SGD :565-575, _adam_update :719-770
//
// Rollout buffers are time-major [T, B] (board index contiguous) so that every per-step kernel and
// the per-board scans are fully coalesced.
#include <cuda_runtime.h>

#include <vector>

#include "b2048_horizon.cuh"
#include "b2048_internal.h"
#include "b2048_mlp.cuh"

namespace b2 {

// ------------------------------------------------------------------------------------------------ K4
// One thread per board, sequential in t (the recurrence is evaluated in float64 with separately
// rounded multiply and add exactly like the reference's Python loop, then stored as float32).
__global__ void __launch_bounds__(256) reverse_scan_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                            const int32_t* __restrict__ len, double c, int T, int64_t B) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int L = len ? min(len[b], T) : T;
    double G = 0.0;
    for (int t = T - 1; t >= L; --t) y[(int64_t)t * B + b] = 0.0f;
    for (int t = L - 1; t >= 0; --t) {
        G = __dadd_rn((double)x[(int64_t)t * B + b], __dmul_rn(c, G));
        y[(int64_t)t * B + b] = (float)G;
    }
}

// Small batches: one warp per board, 32 timesteps per pass, suffix scan of the affine maps
// G -> x_t + c G composed with warp shuffles (float32; within 1e-3 relative of the float64 loop).
__global__ void __launch_bounds__(256) reverse_scan_warp_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                                 const int32_t* __restrict__ len, float c, int T,
                                                                 int64_t B) {
    int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    int lane = threadIdx.x & 31;
    if (b >= B) return;
    int L = len ? min(len[b], T) : T;
    float carry = 0.0f;  // G at the start of the already-processed suffix
    for (int t0 = ((T - 1) / 32) * 32; t0 >= 0; t0 -= 32) {
        int t = t0 + lane;
        bool live = t < L;
        // element = affine map (m, a): G_t = a + m * G_{t+1}
        float a = live ? x[(int64_t)t * B + b] : 0.0f;
        float m = live ? c : 0.0f;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            float a2 = __shfl_down_sync(0xFFFFFFFFu, a, d);
            float m2 = __shfl_down_sync(0xFFFFFFFFu, m, d);
            if (lane + d < 32) { a = fmaf(m, a2, a); m = m * m2; }
        }
        float g = fmaf(m, carry, a);
        if (t < T) y[(int64_t)t * B + b] = live ? g : 0.0f;
        carry = __shfl_sync(0xFFFFFFFFu, g, 0);
    }
}

// ------------------------------------------------------------------------------------------------ K5
// Single pass: acc[0] += sum w, acc[1] += sum w*v, acc[2] += sum w*v*v, acc[3] += count (float64
// accumulators; the weighted variance is acc[2]/acc[0] - mean^2).  Being plain sums, the four numbers
// can be all-reduced across ranks before the advantages are formed.
__global__ void __launch_bounds__(256) weighted_stats_kernel(const float* __restrict__ v, const int32_t* __restrict__ len,
                                                              const float* __restrict__ w, int T, int64_t B,
                                                              double* __restrict__ acc) {
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    const int64_t total = (int64_t)T * B;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t b = i % B;
        int t = (int)(i / B);
        int L = len ? len[b] : T;
        if (t < L) {
            double wb = w ? (double)w[b] : 1.0;
            double val = (double)v[i];
            s0 += wb; s1 += wb * val; s2 += wb * val * val; s3 += 1.0;
        }
    }
    for (int d = 16; d > 0; d >>= 1) {
        s0 += __shfl_down_sync(0xFFFFFFFFu, s0, d); s1 += __shfl_down_sync(0xFFFFFFFFu, s1, d);
        s2 += __shfl_down_sync(0xFFFFFFFFu, s2, d); s3 += __shfl_down_sync(0xFFFFFFFFu, s3, d);
    }
    __shared__ double sh[4][8];
    int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { sh[0][warp] = s0; sh[1][warp] = s1; sh[2][warp] = s2; sh[3][warp] = s3; }
    __syncthreads();
    if (threadIdx.x < 4) {
        double s = 0.0;
        for (int k = 0; k < 8; ++k) s += sh[threadIdx.x][k];
        if (s != 0.0) atomicAdd(acc + threadIdx.x, s);
    }
}

// adv[t,b] per baseline mode; coef[t,b] = adv * w_b / (len_b * n_traj)   (0 beyond the episode end)
//   mode 0 off, 1 each (per-episode mean, needs ep_mean[b]), 2 batch, 3 batch_norm (stats in acc)
__global__ void __launch_bounds__(256) advantage_kernel(const float* __restrict__ v, const int32_t* __restrict__ len,
                                                         const float* __restrict__ w, const float* __restrict__ ep_mean,
                                                         const double* __restrict__ acc, int mode, float n_traj, int T,
                                                         int64_t B, float* __restrict__ adv, float* __restrict__ coef) {
    float mean = 0.0f, stdv = 1.0f;
    if (mode >= 2) {
        double sw = acc[0];
        if (sw < 1e-8) { mean = 0.0f; stdv = 1.0f; }       // reinforce_agent.py:874-875
        else {
            double m = acc[1] / sw, var = acc[2] / sw - m * m;
            mean = (float)m;
            stdv = (float)sqrt(var > 0.0 ? var : 0.0);
        }
        if (stdv < 1e-8f) stdv = 1e-8f;                      // reinforce_agent.py:319-320
    }
    const int64_t total = (int64_t)T * B;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t b = i % B;
        int t = (int)(i / B);
        int L = len ? len[b] : T;
        float a = 0.0f, cf = 0.0f;
        if (t < L) {
            float val = v[i];
            if (mode == 0) a = val;
            else if (mode == 1) a = val - ep_mean[b];
            else if (mode == 2) a = val - mean;
            else a = (val - mean) / stdv;
            float wb = w ? w[b] : 1.0f;
            cf = a * (wb * (1.0f / ((float)L * n_traj)));
        }
        if (adv) adv[i] = a;
        if (coef) coef[i] = cf;
    }
}

// ------------------------------------------------------------------------------------------------ fixed-horizon windows
// advantage_kernel's modes 0 / 2 / 3 for a fixed-horizon window: the samples of lane b are t < valid_len[b] and the divisor
// is T n_traj (an episode's length is not known inside the window).  A kernel of its own so that advantage_kernel's code
// stays as it is.
__global__ void __launch_bounds__(256) advantage_window_kernel(const float* __restrict__ v, const int32_t* __restrict__ valid_len,
                                                                const double* __restrict__ acc, int mode, float n_traj,
                                                                int T, int64_t B, float* __restrict__ adv,
                                                                float* __restrict__ coef) {
    float mean = 0.0f, stdv = 1.0f;
    if (mode >= 2) {                                         // same statistics as advantage_kernel
        double sw = acc[0];
        if (sw >= 1e-8) {
            double m = acc[1] / sw, var = acc[2] / sw - m * m;
            mean = (float)m;
            stdv = (float)sqrt(var > 0.0 ? var : 0.0);
        }
        if (stdv < 1e-8f) stdv = 1e-8f;
    }
    const float inv = 1.0f / ((float)T * n_traj);
    const int64_t total = (int64_t)T * B;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int t = (int)(i / B);
        float a = 0.0f, cf = 0.0f;
        if (t < valid_len[i % B]) {
            const float val = v[i];
            a = mode == 0 ? val : (mode == 2 ? val - mean : (val - mean) / stdv);
            cf = a * inv;
        }
        adv[i] = a;
        coef[i] = cf;
    }
}

// One thread per lane, reverse in t (segment_lane, b2048_horizon.cuh).
__global__ void __launch_bounds__(256) segment_targets_kernel(const float* __restrict__ reward, const uint8_t* __restrict__ flags,
                                                               const float* __restrict__ value, float gamma, double c,
                                                               int huber, float huber_delta, float inv_div, int T, int64_t B,
                                                               float* __restrict__ v, float* __restrict__ td,
                                                               float* __restrict__ gcoef, int32_t* __restrict__ valid_len) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    valid_len[b] = segment_lane(reward + b, flags + b, value ? value + b : nullptr, B, T, gamma, c, huber, huber_delta,
                                inv_div, v + b, td ? td + b : nullptr, gcoef ? gcoef + b : nullptr);
}

__device__ __forceinline__ void atomic_max_f64(double* a, double v) {
    unsigned long long* p = reinterpret_cast<unsigned long long*>(a);
    unsigned long long old = *p;
    while (__longlong_as_double(old) < v) {
        const unsigned long long prev = atomicCAS(p, old, (unsigned long long)__double_as_longlong(v));
        if (prev == old) break;
        old = prev;
    }
}
__device__ __forceinline__ void atomic_min_f64(double* a, double v) {
    unsigned long long* p = reinterpret_cast<unsigned long long*>(a);
    unsigned long long old = *p;
    while (__longlong_as_double(old) > v) {
        const unsigned long long prev = atomicCAS(p, old, (unsigned long long)__double_as_longlong(v));
        if (prev == old) break;
        old = prev;
    }
}

// Episodes completed inside a window: ep_return[b] carries the undiscounted return of the lane's running episode
// across windows (float64); at each boundary the episode is added to acc = {count, sum, max, min, hist[17] by max-tile
// exponent}.  One thread per lane; per block, register / shared-memory partials and one set of global atomics.
__global__ void __launch_bounds__(256) horizon_episodes_kernel(const float* __restrict__ reward, const uint8_t* __restrict__ flags,
                                                                const uint64_t* __restrict__ board,
                                                                const uint8_t* __restrict__ action,
                                                                const uint16_t* __restrict__ lut_left,
                                                                const uint8_t* __restrict__ lut_merge, int T, int64_t B,
                                                                double* __restrict__ ep_return, double* __restrict__ acc) {
    __shared__ unsigned hist[17];
    __shared__ double part[4][8];
    if (threadIdx.x < 17) hist[threadIdx.x] = 0u;
    __syncthreads();
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double n = 0.0, sum = 0.0, mx = -INFINITY, mn = INFINITY;
    if (b < B) {
        double carry = ep_return[b];
        for (int t = 0; t < T; ++t) {
            const int64_t i = (int64_t)t * B + b;
            carry += (double)reward[i];
            if (flags[i + B] & (B2048_F_DONE | B2048_F_TRUNC)) {
                n += 1.0;
                sum += carry;
                mx = fmax(mx, carry);
                mn = fmin(mn, carry);
                atomicAdd(&hist[final_max_exp(board[i], action[i], lut_left, lut_merge)], 1u);
                carry = 0.0;
            }
        }
        ep_return[b] = carry;
    }
    for (int d = 16; d > 0; d >>= 1) {
        n += __shfl_down_sync(0xFFFFFFFFu, n, d); sum += __shfl_down_sync(0xFFFFFFFFu, sum, d);
        mx = fmax(mx, __shfl_down_sync(0xFFFFFFFFu, mx, d)); mn = fmin(mn, __shfl_down_sync(0xFFFFFFFFu, mn, d));
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { part[0][warp] = n; part[1][warp] = sum; part[2][warp] = mx; part[3][warp] = mn; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int k = 1; k < 8; ++k) {
            n += part[0][k]; sum += part[1][k]; mx = fmax(mx, part[2][k]); mn = fmin(mn, part[3][k]);
        }
        if (n != 0.0) {
            atomicAdd(acc + 0, n);
            atomicAdd(acc + 1, sum);
            atomic_max_f64(acc + 2, mx);
            atomic_min_f64(acc + 3, mn);
        }
    }
    if (threadIdx.x < 17 && hist[threadIdx.x] != 0u) atomicAdd(acc + 4 + threadIdx.x, (double)hist[threadIdx.x]);
}

// One thread per listed slot s = t B + b of a window: the board lane b was cut on by step t (pre_reset_board: step_one
// with auto-reset off at the rollout's counter t0 + t + 1).
__global__ void __launch_bounds__(256) replay_pre_reset_kernel(const uint64_t* __restrict__ board, const uint8_t* __restrict__ action,
                                                                const int64_t* __restrict__ slots, int64_t K, int64_t B,
                                                                uint64_t seed, uint64_t gid0, uint32_t t0,
                                                                const uint16_t* __restrict__ lut_left,
                                                                const uint8_t* __restrict__ lut_merge, uint64_t* __restrict__ out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const int64_t s = slots[k];
    const int64_t t = s / B, b = s - t * B;
    out[k] = pre_reset_board(board[s], action[s], seed, gid0 + (uint64_t)b, t0 + (uint32_t)t + 1u, lut_left, lut_merge);
}

// out[slots[k]] = reward[slots[k]] + gamma value[k] (fold_bootstrap); the other elements are copied by the launcher.
// (reward and out may be the same buffer)
__global__ void __launch_bounds__(256) fold_bootstrap_kernel(const float* reward, const int64_t* __restrict__ slots,
                                                              const float* __restrict__ value, int64_t K, float gamma, float* out) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const int64_t s = slots[k];
    out[s] = fold_bootstrap(reward[s], gamma, value[k]);
}

// The slot list lives on the device: copy it to the host and check every index against [lo, hi).
static int check_slots(const int64_t* slots, int64_t K, int64_t lo, int64_t hi, cudaStream_t s, const char* who) {
    std::vector<int64_t> host((size_t)K);
    B2_CUDA(cudaMemcpyAsync(host.data(), slots, (size_t)K * sizeof(int64_t), cudaMemcpyDefault, s));
    B2_CUDA(cudaStreamSynchronize(s));
    for (int64_t k = 0; k < K; ++k)
        if (host[(size_t)k] < lo || host[(size_t)k] >= hi)
            return fail(B2048_ERR_INVALID, std::string(who) + ": slot " + std::to_string(host[(size_t)k]) + " at index " +
                                               std::to_string(k) + " is outside [" + std::to_string(lo) + ", " +
                                               std::to_string(hi) + ")");
    return B2048_OK;
}

// per-episode mean of v over t < len (baseline "each", reinforce_agent.py:296-302)
__global__ void __launch_bounds__(256) episode_mean_kernel(const float* __restrict__ v, const int32_t* __restrict__ len,
                                                            int T, int64_t B, float* __restrict__ ep_mean) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    int L = len ? min(len[b], T) : T;
    float s = 0.0f;
    for (int t = 0; t < L; ++t) s += v[(int64_t)t * B + b];
    ep_mean[b] = L > 0 ? s / (float)L : 0.0f;
}

// TD(0): delta = r + gamma * V(s_{t+1}) * [t+1 < len] - V(s_t)   (reinforce_agent.py:439-447)
// gcoef = dLoss/dV * w_b/(len_b n_traj), dLoss/dV = -delta (mse) or clip(-delta, +-huber) (reinforce_agent.py:884-910)
__global__ void __launch_bounds__(256) td_error_kernel(const float* __restrict__ reward, const float* __restrict__ value,
                                                        const int32_t* __restrict__ len, const float* __restrict__ w,
                                                        float gamma, int huber, float huber_delta, float n_traj, int T,
                                                        int64_t B, float* __restrict__ td, float* __restrict__ gcoef) {
    const int64_t total = (int64_t)T * B;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        int64_t b = i % B;
        int t = (int)(i / B);
        int L = len ? len[b] : T;
        float d = 0.0f, g = 0.0f;
        if (t < L) {
            float vn = (t + 1 < L) ? value[i + B] : 0.0f;
            float target = reward[i] + gamma * vn;
            float vc = value[i];
            d = target - vc;
            float diff = vc - target;
            g = diff;
            if (huber && fabsf(diff) > huber_delta) g = diff > 0.0f ? huber_delta : (diff < 0.0f ? -huber_delta : 0.0f);
            float wb = w ? w[b] : 1.0f;
            g *= wb * (1.0f / ((float)L * n_traj));
        }
        td[i] = d;
        if (gcoef) gcoef[i] = g;
    }
}

// ------------------------------------------------------------------------------------------------ K6 phase A
struct BackwardArgs {
    MlpDev mlp;
    const float* WT[B2048_MAX_LAYERS];  // transposed hidden weights, WT[l] = W[l]^T as [dims[l+1]][dims[l]] (l >= 1)
    const uint64_t* board;
    const uint8_t* mask_flags;
    const uint8_t* action;
    const float* coef;
    float* gact[B2048_MAX_LAYERS];   // out: a_l  [n][dims[l]]   for l = 1..L-1
    float* gdelta[B2048_MAX_LAYERS]; // out: d_l  [n][dims[l+1]] for l = 0..L-1 (gradient wrt layer-l pre-activation)
    int64_t n;
    int head_mode;                   // 0: actor, d_L = coef * (onehot(a) - pi);  1: value head, d_L = coef
};

__global__ void __launch_bounds__(kMlpThreads, 1) mlp_backward_kernel(const __grid_constant__ BackwardArgs args) {
    extern __shared__ __align__(16) float arena[];
    const MlpDev& m = args.mlp;
    const int L = m.n_layers;
    const int n_out = m.dims[L];
    float* dh = arena + act_offset(m.dims, L);  // [kTileM][4] head deltas
    const int64_t n_tiles = (args.n + kTileM - 1) / kTileM;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t s0 = tile * kTileM;
        tile_forward_hidden(arena, m, args.board, s0, args.n, const_cast<float* const*>(args.gact));
        float out = tile_head(arena, m);
        const int b = threadIdx.x >> 2, j = threadIdx.x & 3;
        const int64_t s = s0 + b;
        const bool valid = s < args.n;
        float cf = valid ? args.coef[s] : 0.0f;
        float d;
        if (args.head_mode == 0) {
            uint32_t fl = 0xFu;
            const bool use_mask = args.mask_flags != nullptr;
            if (use_mask && valid) fl = args.mask_flags[s];
            if (j >= n_out) out = -INFINITY;
            float p = quad_softmax(out, (fl >> j) & 1u, use_mask);
            uint32_t a = valid ? args.action[s] : 0u;
            d = cf * ((a == (uint32_t)j ? 1.0f : 0.0f) - p);  // reinforce_agent.py:340-344
        } else {
            d = cf;
        }
        if (j >= n_out) d = 0.0f;
        dh[b * 4 + j] = d;
        if (valid && j < n_out) args.gdelta[L - 1][s * n_out + j] = d;
        __syncthreads();
        // back through the head: d_{L-2}[b][i] = (sum_j d_{L-1}[b][j] W_{L-1}[i][j]) * act'(a_{L-1}[b][i])
        if (L >= 2) {
            const int K = m.dims[L - 1];
            float* a_prev = arena + act_offset(m.dims, L - 1);
            const int stride = act_stride(m.dims, L - 1);
            const float* Wl = m.W[L - 1];
            for (int idx = threadIdx.x; idx < kTileM * K; idx += kMlpThreads) {
                int bb = idx / K, i = idx - bb * K;
                float acc = 0.0f;
                for (int jj = 0; jj < n_out; ++jj) acc = fmaf(dh[bb * 4 + jj], __ldg(Wl + (size_t)i * n_out + jj), acc);
                float v = acc * activate_grad(a_prev[bb * stride + i], m.activation);
                a_prev[bb * stride + i] = v;
                if (s0 + bb < args.n) args.gdelta[L - 2][(s0 + bb) * K + i] = v;
            }
            __syncthreads();
            // remaining hidden layers: same register-tiled product with the transposed weights
            for (int l = L - 2; l >= 1; --l) {
                float* din = arena + act_offset(m.dims, l + 1);   // holds d_l  [M][dims[l+1]]
                float* dout = arena + act_offset(m.dims, l);      // holds a_l, becomes d_{l-1}
                tile_layer<1>(din, m.dims[l + 1], act_stride(m.dims, l + 1), args.WT[l], nullptr, m.dims[l], dout,
                              act_stride(m.dims, l), m.activation, false, args.gdelta[l - 1], s0, args.n);
                __syncthreads();
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------------ K6 phase B
// C[Mi x N] += sum_s A[s][Mi] * D[s][N].  64 x 64 output tile per CTA, 256 threads x (4 x 4), split over samples
// in gridDim.z chunks; partial tiles are reduced with float atomics into the (pre-zeroed) gradient.
// a_mode: 0 = A read from memory [n][Mi]; 1/2/3 = A generated from packed boards (raw / log2 / onehot input).
__global__ void __launch_bounds__(256) atb_kernel(const float* __restrict__ A, const uint64_t* __restrict__ board, int a_mode,
                                                   float obs_scale, const float* __restrict__ D, float* __restrict__ C,
                                                   int Mi, int N, int64_t n, int64_t chunk) {
    __shared__ float As[32][64 + 4];
    __shared__ float Ds[32][64 + 4];
    const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
    const int64_t s_begin = (int64_t)blockIdx.z * chunk;
    const int64_t s_end = min(n, s_begin + chunk);
    const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
    for (int64_t s0 = s_begin; s0 < s_end; s0 += 32) {
        for (int idx = threadIdx.x; idx < 32 * 64; idx += 256) {
            int k = idx >> 6, c = idx & 63;
            int64_t s = s0 + k;
            float av = 0.0f, dv = 0.0f;
            if (s < s_end) {
                int mi = m0 + c;
                if (mi < Mi) {
                    if (a_mode == 0) av = A[s * Mi + mi];
                    else {
                        uint64_t bd = board[s];
                        if (a_mode == B2048_OBS_ONEHOT) {
                            int cell = mi / 17, ch = mi - 17 * cell;
                            av = ((int)((bd >> (4 * cell)) & 0xFull) == ch) ? 1.0f : 0.0f;
                        } else {
                            uint32_t e = (uint32_t)((bd >> (4 * mi)) & 0xFull);
                            av = a_mode == B2048_OBS_RAW ? (e ? (float)(1u << e) : 0.0f) : (float)e * obs_scale;
                        }
                    }
                }
                int ni = n0 + c;
                if (ni < N) dv = D[s * N + ni];
            }
            As[k][c] = av;
            Ds[k][c] = dv;
        }
        __syncthreads();
#pragma unroll 8
        for (int k = 0; k < 32; ++k) {
            float4 a = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
            float4 d = *reinterpret_cast<const float4*>(&Ds[k][tx * 4]);
            float av[4] = {a.x, a.y, a.z, a.w}, dv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
            for (int i = 0; i < 4; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], dv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            int mi = m0 + ty * 4 + i, ni = n0 + tx * 4 + j;
            if (mi < Mi && ni < N && acc[i][j] != 0.0f) atomicAdd(C + (size_t)mi * N + ni, acc[i][j]);
        }
}

__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ D, float* __restrict__ out, int N, int64_t n,
                                                      int64_t chunk) {
    const int64_t s_begin = (int64_t)blockIdx.y * chunk, s_end = min(n, s_begin + chunk);
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < N; c += gridDim.x * blockDim.x) {
        float s = 0.0f;
        for (int64_t r = s_begin; r < s_end; ++r) s += D[r * N + c];
        if (s != 0.0f) atomicAdd(out + c, s);
    }
}

__global__ void transpose_kernel(const float* __restrict__ in, float* __restrict__ out, int rows, int cols) {
    __shared__ float tile[32][33];
    int x = blockIdx.x * 32 + threadIdx.x, y0 = blockIdx.y * 32;
    for (int j = threadIdx.y; j < 32; j += blockDim.y)
        if (x < cols && y0 + j < rows) tile[j][threadIdx.x] = in[(size_t)(y0 + j) * cols + x];
    __syncthreads();
    int xo = blockIdx.y * 32 + threadIdx.x, yo0 = blockIdx.x * 32;
    for (int j = threadIdx.y; j < 32; j += blockDim.y)
        if (xo < rows && yo0 + j < cols) out[(size_t)(yo0 + j) * rows + xo] = tile[threadIdx.x][j];
}

// ------------------------------------------------------------------------------------------------ optimiser
__global__ void __launch_bounds__(256) sumsq_kernel(const float* __restrict__ g, int64_t n, double* __restrict__ out) {
    double s = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        double v = (double)g[i];
        s += v * v;
    }
    for (int d = 16; d > 0; d >>= 1) s += __shfl_down_sync(0xFFFFFFFFu, s, d);
    __shared__ double sh[8];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int k = 0; k < 8; ++k) t += sh[k];
        atomicAdd(out, t);
    }
}

// clip_coef = max_norm / max(norm, 1e-8), applied only if < 1 (reinforce_agent.py:849-855)
__device__ __forceinline__ float clip_coef(const double* sumsq, float max_norm) {
    float norm = (float)sqrt(*sumsq);
    float coef = max_norm / fmaxf(norm, 1e-8f);
    return coef < 1.0f ? coef : 1.0f;
}

// theta += sign * lr * clip(g)   (actor: ascent sign=+1; critic: descent sign=-1, reinforce_agent.py:565-575)
__global__ void __launch_bounds__(256) sgd_kernel(float* __restrict__ theta, float* __restrict__ g, int64_t n,
                                                   const double* __restrict__ sumsq, float max_norm, float lr, float sign) {
    float cc = clip_coef(sumsq, max_norm);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float gv = g[i] * cc;
        g[i] = gv;
        theta[i] += sign * lr * gv;
    }
}

// _adam_update (reinforce_agent.py:719-770), t = step count after increment
__global__ void __launch_bounds__(256) adam_kernel(float* __restrict__ theta, float* __restrict__ g, float* __restrict__ m,
                                                    float* __restrict__ v, int64_t n, const double* __restrict__ sumsq,
                                                    float max_norm, float lr, float sign, float beta1, float beta2,
                                                    float bc1, float bc2) {
    float cc = clip_coef(sumsq, max_norm);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        float gv = g[i] * cc;
        g[i] = gv;
        float mi = beta1 * m[i] + (1.0f - beta1) * gv;
        float vi = beta2 * v[i] + (1.0f - beta2) * (gv * gv);
        m[i] = mi;
        v[i] = vi;
        float mh = mi / bc1, vh = vi / bc2;
        theta[i] = theta[i] + sign * lr * mh / (sqrtf(vh) + 1e-8f);
    }
}

static int ew_grid(int64_t n, int num_sms) {
    int64_t b = (n + 255) / 256;
    int64_t cap = (int64_t)num_sms * 8;
    return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

}  // namespace b2

using namespace b2;

extern "C" int b2048_reverse_scan(const float* x, float* y, const int32_t* len, float c, int32_t T, int64_t B,
                                  void* stream) {
    B2_REQUIRE(T >= 0 && B >= 0, "b2048_reverse_scan: negative size");
    if (T == 0 || B == 0) return B2048_OK;
    B2_REQUIRE(x && y, "b2048_reverse_scan: x/y is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    if (B >= 2048) {
        reverse_scan_kernel<<<(unsigned)((B + 255) / 256), 256, 0, s>>>(x, y, len, (double)c, T, B);
    } else {
        reverse_scan_warp_kernel<<<(unsigned)((B * 32 + 255) / 256), 256, 0, s>>>(x, y, len, c, T, B);
    }
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_reverse_scan_f64(const float* x, float* y, const int32_t* len, double c, int32_t T, int64_t B,
                                      void* stream) {
    B2_REQUIRE(T >= 0 && B >= 0, "b2048_reverse_scan_f64: negative size");
    if (T == 0 || B == 0) return B2048_OK;
    B2_REQUIRE(x && y, "b2048_reverse_scan_f64: x/y is NULL");
    reverse_scan_kernel<<<(unsigned)((B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, y, len, c, T, B);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_advantages(b2048_handle* h, const float* v, const int32_t* len, const float* ep_weight,
                                int32_t baseline_mode, float n_traj, int32_t T, int64_t B, float* adv, float* coef,
                                double* stats /* device, 4 doubles */, int32_t stats_precomputed,
                                float* ep_mean_scratch /* [B] */, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_advantages: handle is NULL");
    B2_REQUIRE(baseline_mode >= 0 && baseline_mode <= 3, "b2048_advantages: unknown baseline mode");  // reinforce_agent.py:325
    B2_REQUIRE(T >= 0 && B >= 0, "b2048_advantages: negative size");
    if (T == 0 || B == 0) return B2048_OK;
    B2_REQUIRE(v && stats, "b2048_advantages: v/stats is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t total = (int64_t)T * B;
    if (baseline_mode >= 2 && !stats_precomputed) {
        B2_CUDA(cudaMemsetAsync(stats, 0, 4 * sizeof(double), s));
        weighted_stats_kernel<<<ew_grid(total, h->num_sms), 256, 0, s>>>(v, len, ep_weight, T, B, stats);
    } else if (baseline_mode == 1) {
        B2_REQUIRE(ep_mean_scratch != nullptr, "b2048_advantages: ep_mean_scratch required for baseline 'each'");
        episode_mean_kernel<<<(unsigned)((B + 255) / 256), 256, 0, s>>>(v, len, T, B, ep_mean_scratch);
    }
    advantage_kernel<<<ew_grid(total, h->num_sms), 256, 0, s>>>(v, len, ep_weight, ep_mean_scratch, stats, baseline_mode,
                                                                 n_traj, T, B, adv, coef);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

// The sums behind the "batch" / "batch_norm" baselines, ADDED into stats[0..3] (zero it first): callers that
// shard episodes over ranks all-reduce the four doubles and then call b2048_advantages(stats_precomputed=1).
extern "C" int b2048_weighted_stats(b2048_handle* h, const float* v, const int32_t* len, const float* ep_weight,
                                    int32_t T, int64_t B, double* stats, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_weighted_stats: handle is NULL");
    B2_REQUIRE(T >= 0 && B >= 0, "b2048_weighted_stats: negative size");
    if (T == 0 || B == 0) return B2048_OK;
    B2_REQUIRE(v && stats, "b2048_weighted_stats: v/stats is NULL");
    weighted_stats_kernel<<<ew_grid((int64_t)T * B, h->num_sms), 256, 0, (cudaStream_t)stream>>>(v, len, ep_weight, T, B,
                                                                                               stats);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_td_errors(b2048_handle* h, const float* reward, const float* value, const int32_t* len,
                               const float* ep_weight, float gamma, int32_t huber, float huber_delta, float n_traj,
                               int32_t T, int64_t B, float* td, float* gcoef, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_td_errors: handle is NULL");
    B2_REQUIRE(T >= 0 && B >= 0, "b2048_td_errors: negative size");
    if (T == 0 || B == 0) return B2048_OK;
    B2_REQUIRE(reward && value && td, "b2048_td_errors: NULL buffer");
    td_error_kernel<<<ew_grid((int64_t)T * B, h->num_sms), 256, 0, (cudaStream_t)stream>>>(
        reward, value, len, ep_weight, gamma, huber, huber_delta, n_traj, T, B, td, gcoef);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_segment_targets(b2048_handle* h, const float* reward, const uint8_t* flags, const float* value,
                                     double gamma, double lambda, int32_t huber, float huber_delta, float n_traj, int32_t T,
                                     int64_t B, float* v, float* td, float* gcoef, int32_t* valid_len, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_segment_targets: handle is NULL");
    B2_REQUIRE(T >= 0 && B >= 0, "b2048_segment_targets: negative size");
    if (T == 0 || B == 0) return B2048_OK;
    B2_REQUIRE(reward && flags && v && valid_len, "b2048_segment_targets: NULL buffer");
    B2_REQUIRE(!value || (td && gcoef), "b2048_segment_targets: td and gcoef are required with values");
    B2_REQUIRE(n_traj > 0.0f, "b2048_segment_targets: n_traj must be positive");
    const double c = value ? gamma * lambda : gamma;
    const float inv_div = 1.0f / ((float)T * n_traj);
    segment_targets_kernel<<<(unsigned)((B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reward, flags, value, (float)gamma, c, huber, huber_delta, inv_div, T, B, v, value ? td : nullptr,
        value ? gcoef : nullptr, valid_len);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_advantages_window(b2048_handle* h, const float* v, const int32_t* valid_len, int32_t baseline_mode,
                                       float n_traj, int32_t T, int64_t B, float* adv, float* coef, double* stats,
                                       int32_t stats_precomputed, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_advantages_window: handle is NULL");
    B2_REQUIRE(baseline_mode == 0 || baseline_mode == 2 || baseline_mode == 3,
               "b2048_advantages_window: baseline mode must be 0 (off), 2 (batch) or 3 (batch_norm)");
    B2_REQUIRE(T >= 0 && B >= 0, "b2048_advantages_window: negative size");
    if (T == 0 || B == 0) return B2048_OK;
    B2_REQUIRE(v && valid_len && stats, "b2048_advantages_window: v/valid_len/stats is NULL");
    cudaStream_t s = (cudaStream_t)stream;
    const int64_t total = (int64_t)T * B;
    if (baseline_mode >= 2 && !stats_precomputed) {
        B2_CUDA(cudaMemsetAsync(stats, 0, 4 * sizeof(double), s));
        weighted_stats_kernel<<<ew_grid(total, h->num_sms), 256, 0, s>>>(v, valid_len, nullptr, T, B, stats);
    }
    advantage_window_kernel<<<ew_grid(total, h->num_sms), 256, 0, s>>>(v, valid_len, stats, baseline_mode, n_traj, T, B,
                                                                        adv, coef);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_horizon_episodes(b2048_handle* h, const float* reward, const uint8_t* flags, const uint64_t* board,
                                      const uint8_t* action, int32_t T, int64_t B, double* ep_return, double* stats,
                                      void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_horizon_episodes: handle is NULL");
    B2_REQUIRE(T >= 0 && B >= 0, "b2048_horizon_episodes: negative size");
    if (T == 0 || B == 0) return B2048_OK;
    B2_REQUIRE(reward && flags && board && action && ep_return && stats, "b2048_horizon_episodes: NULL buffer");
    horizon_episodes_kernel<<<(unsigned)((B + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
        reward, flags, board, action, lut_left_ptr(h), lut_merge_ptr(h), T, B, ep_return, stats);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_replay_pre_reset(b2048_handle* h, const uint64_t* boards, const uint8_t* actions, const int64_t* slots,
                                      int64_t K, int64_t B, uint64_t seed, uint64_t gid0, uint32_t t0, uint64_t* out,
                                      void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_replay_pre_reset: handle is NULL");
    B2_REQUIRE(K >= 0 && B >= 0, "b2048_replay_pre_reset: negative size");
    if (K == 0) return B2048_OK;
    B2_REQUIRE(B > 0, "b2048_replay_pre_reset: slots listed for a window of no lanes");
    B2_REQUIRE(boards && actions && slots && out, "b2048_replay_pre_reset: NULL buffer");
    cudaStream_t s = (cudaStream_t)stream;
    // the window's length is not an argument: only the lower bound of the slots can be checked
    int st = check_slots(slots, K, 0, INT64_MAX, s, "b2048_replay_pre_reset");
    if (st != B2048_OK) return st;
    replay_pre_reset_kernel<<<(unsigned)((K + 255) / 256), 256, 0, s>>>(boards, actions, slots, K, B, seed, gid0, t0,
                                                                          lut_left_ptr(h), lut_merge_ptr(h), out);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_fold_bootstrap(b2048_handle* h, const float* reward, const int64_t* slots, const float* value, int64_t K,
                                    int64_t n, float gamma, float* reward_out, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_fold_bootstrap: handle is NULL");
    B2_REQUIRE(K >= 0 && n >= 0, "b2048_fold_bootstrap: negative size");
    if (n == 0 && K == 0) return B2048_OK;
    B2_REQUIRE(reward && reward_out && (K == 0 || (slots && value)), "b2048_fold_bootstrap: NULL buffer");
    cudaStream_t s = (cudaStream_t)stream;
    if (K > 0) {
        int st = check_slots(slots, K, 0, n, s, "b2048_fold_bootstrap");
        if (st != B2048_OK) return st;
    }
    if (reward_out != reward) B2_CUDA(cudaMemcpyAsync(reward_out, reward, (size_t)n * sizeof(float), cudaMemcpyDeviceToDevice, s));
    if (K > 0)
        fold_bootstrap_kernel<<<(unsigned)((K + 255) / 256), 256, 0, s>>>(reward, slots, value, K, gamma, reward_out);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int64_t b2048_backward_workspace_floats(const b2048_mlp_desc* mlp, int64_t chunk) {
    if (!mlp || chunk <= 0) return 0;
    int64_t per = 0;
    for (int l = 1; l < mlp->n_layers; ++l) per += 2 * (int64_t)mlp->dims[l];  // a_l and d_{l-1}
    per += mlp->dims[mlp->n_layers];                                            // d_{L-1}
    int64_t wt = 0;
    for (int l = 1; l + 1 < mlp->n_layers; ++l) wt += (int64_t)mlp->dims[l] * mlp->dims[l + 1];
    int64_t floats = per * chunk + wt + 64;
    // the tensor-core paths carve their images out of the same workspace
    if (is_16_256_256(mlp)) {
        const int64_t tc = (backward_tc_workspace_bytes(chunk) + 3) / 4, hp = (backward_hp_workspace_bytes(chunk) + 3) / 4;
        floats = floats > tc ? floats : tc;
        floats = floats > hp ? floats : hp;
    } else if (gen_shape_ok(mlp)) {
        const int64_t gn = (gen_workspace_bytes(mlp, chunk) + 3) / 4;
        floats = floats > gn ? floats : gn;
    }
    return floats;
}

// Accumulates into grads (flat, same layout as the flat parameter vector: W_0, b_0, W_1, b_1, ...):
//   head_mode 0: d/dtheta sum_s coef[s] * log pi(action[s] | board[s])        (policy gradient, ascent direction)
//   head_mode 1: d/dtheta sum_s coef[s] * V(board[s])                          (value head; coef = dLoss/dV * weight)
extern "C" int b2048_mlp_backward(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags,
                                  const uint8_t* action, const float* coef, const b2048_mlp_desc* mlp, float* grads,
                                  int64_t n, int32_t head_mode, float* workspace, int64_t workspace_floats,
                                  int64_t chunk, int32_t precision, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_mlp_backward: handle is NULL");
    B2_REQUIRE(n >= 0, "b2048_mlp_backward: n < 0");
    if (n == 0) return B2048_OK;
    B2_REQUIRE(board && coef && grads && workspace, "b2048_mlp_backward: NULL buffer");
    B2_REQUIRE(head_mode == 1 || action != nullptr, "b2048_mlp_backward: action required for the policy head");
    B2_REQUIRE(chunk > 0, "b2048_mlp_backward: chunk must be positive");
    B2_REQUIRE(precision >= 0 && precision <= 3,
               "b2048_mlp_backward: precision must be 0 (fp32), 1 (bf16 tcgen05), 2 (auto) or 3 (split-fp16 tcgen05)");
    if (precision == 2 || precision == 3) {   // float32-grade tensor-core path (what "auto" selects)
        const bool ok = backward_hp_supported(h, mlp) && n >= 4096 &&
                        workspace_floats * 4 >= backward_hp_workspace_bytes(chunk < n ? chunk : n);
        if (ok)
            return launch_backward_hp(h, board, mask_flags, action, coef, mlp, grads, n, head_mode,
                                      reinterpret_cast<uint8_t*>(workspace), workspace_floats * 4 - 1024, chunk < n ? chunk : n,
                                      (cudaStream_t)stream);
        // every other ReLU shape with 64-multiple hidden layers (the reference's documented one-hot [256, 128, 64] network):
        // the shape-generic kernels of b2048_mlp_gen.cu, same arithmetic
        if (!backward_hp_supported(h, mlp) && gen_supported(h, mlp) && n >= 4096 &&
            workspace_floats * 4 >= gen_workspace_bytes(mlp, chunk < n ? chunk : n))
            return launch_backward_gen(h, board, mask_flags, action, coef, mlp, grads, n, head_mode,
                                       reinterpret_cast<uint8_t*>(workspace), chunk < n ? chunk : n, (cudaStream_t)stream);
        if (precision == 3)
            return fail(B2048_ERR_UNSUPPORTED,
                        "b2048_mlp_backward: the split-fp16 tcgen05 path needs a ReLU network with 1-4 hidden layers of 64 / 128 / "
                        "192 / 256 units, log2 or one-hot observations, n >= 4096 and a workspace of "
                        "b2048_backward_workspace_floats()");
    }
    if (precision == 1) {                     // single-bf16 tensor cores: an explicit opt-in (5 % class gradient error)
        const bool ok = backward_tc_supported(h, mlp) && n >= 4096 &&
                        workspace_floats * 4 >= backward_tc_workspace_bytes(chunk < n ? chunk : n);
        if (ok)
            return launch_backward_tc(h, board, mask_flags, action, coef, mlp, grads, n, head_mode,
                                      reinterpret_cast<uint8_t*>(workspace), chunk < n ? chunk : n, (cudaStream_t)stream);
        return fail(B2048_ERR_UNSUPPORTED,
                    "b2048_mlp_backward: the tcgen05 path needs a 16-256-256-(<=4) ReLU network, raw/log2 observations, "
                    "n >= 4096 and a workspace of b2048_backward_workspace_floats()");
    }
    BackwardArgs a;
    size_t smem = 0;
    int st = validate_mlp(mlp, &a.mlp, &smem, h->smem_optin, "b2048_mlp_backward");
    if (st != B2048_OK) return st;
    B2_REQUIRE(workspace_floats >= b2048_backward_workspace_floats(mlp, chunk), "b2048_mlp_backward: workspace too small");
    const int L = a.mlp.n_layers;
    const int* dims = a.mlp.dims;
    cudaStream_t s = (cudaStream_t)stream;
    // carve the workspace
    float* p = workspace;
    for (int l = 0; l < B2048_MAX_LAYERS; ++l) { a.gact[l] = nullptr; a.gdelta[l] = nullptr; a.WT[l] = nullptr; }
    for (int l = 1; l < L; ++l) { a.gact[l] = p; p += chunk * dims[l]; }
    for (int l = 0; l < L; ++l) { a.gdelta[l] = p; p += chunk * dims[l + 1]; }
    for (int l = 1; l + 1 < L; ++l) {
        float* wt = p;
        p += (int64_t)dims[l] * dims[l + 1];
        dim3 blk(32, 8), grd((dims[l + 1] + 31) / 32, (dims[l] + 31) / 32);
        transpose_kernel<<<grd, blk, 0, s>>>(a.mlp.W[l], wt, dims[l], dims[l + 1]);
        a.WT[l] = wt;
    }
    float *gW[B2048_MAX_LAYERS], *gb[B2048_MAX_LAYERS];
    carve_grads(mlp, grads, gW, gb);
    B2_CUDA(cudaFuncSetAttribute(mlp_backward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (int64_t c0 = 0; c0 < n; c0 += chunk) {
        const int64_t cn = (n - c0) < chunk ? (n - c0) : chunk;
        a.board = board + c0;
        a.mask_flags = mask_flags ? mask_flags + c0 : nullptr;
        a.action = action ? action + c0 : nullptr;
        a.coef = coef + c0;
        a.n = cn;
        a.head_mode = head_mode;
        int64_t tiles = (cn + kTileM - 1) / kTileM;
        int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
        mlp_backward_kernel<<<grid, kMlpThreads, smem, s>>>(a);
        for (int l = 0; l < L; ++l) {
            const int Mi = dims[l], N = dims[l + 1];
            int split = (int)((cn + 4095) / 4096);
            int tiles_mn = ((Mi + 63) / 64) * ((N + 63) / 64);
            int max_split = (h->num_sms * 4 + tiles_mn - 1) / tiles_mn;
            if (split > max_split) split = max_split;
            if (split < 1) split = 1;
            int64_t per = ((cn + split - 1) / split + 31) / 32 * 32;
            dim3 grd((N + 63) / 64, (Mi + 63) / 64, (unsigned)((cn + per - 1) / per));
            atb_kernel<<<grd, 256, 0, s>>>(l == 0 ? nullptr : a.gact[l], a.board, l == 0 ? a.mlp.obs_mode : 0,
                                           a.mlp.obs_scale, a.gdelta[l], gW[l], Mi, N, cn, per);
            int csplit = (int)((cn + 2047) / 2048);
            int64_t cper = (cn + csplit - 1) / csplit;
            dim3 cg((N + 255) / 256, (unsigned)csplit);
            colsum_kernel<<<cg, 256, 0, s>>>(a.gdelta[l], gb[l], N, cn, cper);
        }
    }
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

// clip by global norm + optimiser step on a flat parameter vector (actor or critic).
//   optimizer 0 sgd, 1 adam; sign +1 ascent (actor) / -1 descent (critic); adam_t = step count AFTER increment.
//   norm_out (device double[1]) receives the squared global norm of the UNCLIPPED gradient.
extern "C" int b2048_apply_update(b2048_handle* h, float* theta, float* grads, float* adam_m, float* adam_v, int64_t n,
                                  int32_t optimizer, float lr, float sign, float max_grad_norm, float beta1, float beta2,
                                  int32_t adam_t, double* sumsq_out, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_apply_update: handle is NULL");
    B2_REQUIRE(n >= 0, "b2048_apply_update: n < 0");
    B2_REQUIRE(optimizer == 0 || optimizer == 1, "b2048_apply_update: unknown optimizer");  // reinforce_agent.py:581-582
    if (n == 0) return B2048_OK;
    B2_REQUIRE(theta && grads && sumsq_out, "b2048_apply_update: NULL buffer");
    cudaStream_t s = (cudaStream_t)stream;
    B2_CUDA(cudaMemsetAsync(sumsq_out, 0, sizeof(double), s));
    sumsq_kernel<<<ew_grid(n, h->num_sms), 256, 0, s>>>(grads, n, sumsq_out);
    if (optimizer == 0) {
        sgd_kernel<<<ew_grid(n, h->num_sms), 256, 0, s>>>(theta, grads, n, sumsq_out, max_grad_norm, lr, sign);
    } else {
        B2_REQUIRE(adam_m && adam_v && adam_t >= 1, "b2048_apply_update: adam state required");
        float bc1 = 1.0f - powf(beta1, (float)adam_t), bc2 = 1.0f - powf(beta2, (float)adam_t);
        adam_kernel<<<ew_grid(n, h->num_sms), 256, 0, s>>>(theta, grads, adam_m, adam_v, n, sumsq_out, max_grad_norm, lr,
                                                           sign, beta1, beta2, bc1, bc2);
    }
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}
