// b2048_policy.cu — K3 policy_step and the plain MLP forward (fp32 CUDA-core path).
//
//   policy_step_kernel   encode_observation -> forward_logits -> logits_to_probs -> sample / greedy
//                        (src/MLP.py:22-43, :139-196; src/reinforce_agent.py:126-192) fused: the packed
//                        board is the only per-board input, the action byte (+ optional probs / logits)
//                        the only output; activations never leave shared memory.
//   policy_step_np_kernel  the same over a live-board list, sampling rng.choice(4, p) on per-board NumPy streams
//                        (b2048_rollout_many_np: the reference's own seeded episodes)
//   mlp_forward_kernel   forward_logits only (critic values V(s), logits for tests / update)
#include <cuda_runtime.h>

#include "b2048_device.cuh"
#include "b2048_internal.h"
#include "b2048_mlp.cuh"
#include "b2048_np_rng.cuh"

namespace b2 {

struct PolicyArgs {
    MlpDev mlp;
    const uint64_t* board;
    const uint8_t* mask_flags;
    uint8_t* action;
    float* probs;
    float* logits;
    int64_t n;
    uint64_t seed, gid0;
    uint32_t t;
    int greedy;
};

// Extra inputs of the reference-seeded variant policy_step_np_kernel (b2048_rollout_many_np)
struct PolicyNpArgs {
    b2048_np_rng* rng;         // per board: the NumPy policy stream rng.choice draws from, advanced in place
    const int32_t* ep_len;     // a finished board (ep_len != 0) draws nothing and gets no action
    const int32_t* slot_map;   // live-board list: sample s is board slot_map[s] (NULL: board s)
    const int32_t* n_dev;      // with slot_map: the number of listed boards, read on the device
};

// kNp: actions sampled by rng.choice(4, p) on the board's NumPy stream (b2048_np_rng.cuh) over the listed boards; a
// board's probabilities are the same arithmetic whatever its tile or row, so they do not depend on its position.
template <bool kNp>
__device__ __forceinline__ void policy_step_body(const PolicyArgs& args, const PolicyNpArgs& npa) {
    extern __shared__ __align__(16) float arena[];
    const MlpDev& m = args.mlp;
    const int n_out = m.dims[m.n_layers];
    int64_t n = args.n;
    if constexpr (kNp) {
        if (npa.n_dev) n = *npa.n_dev;   // uniform over the grid
    }
    const int64_t n_tiles = (n + kTileM - 1) / kTileM;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t s0 = tile * kTileM;
        tile_forward_hidden(arena, m, args.board, s0, n, nullptr, kNp ? npa.slot_map : nullptr);
        float logit = tile_head(arena, m);
        const int b = threadIdx.x >> 2, j = threadIdx.x & 3;
        int64_t s = s0 + b;
        bool valid = s < n;
        if constexpr (kNp) {
            if (valid && npa.slot_map) s = npa.slot_map[s];
            if (valid && npa.ep_len[s] != 0) valid = false;   // finished: nothing drawn, nothing written
        }
        uint32_t fl = 0xFu;
        const bool use_mask = args.mask_flags != nullptr;
        if (use_mask && valid) fl = args.mask_flags[s];
        const bool legal = (fl >> j) & 1u;
        if (j >= n_out) logit = -INFINITY;  // fewer than 4 outputs: the spare lanes never win
        float p = quad_softmax(logit, legal, use_mask);
        if (valid && j < n_out) {
            if (args.probs) args.probs[s * n_out + j] = p;
            if (args.logits) args.logits[s * n_out + j] = logit;
        }
        // gather the quad's probabilities
        const int qbase = (threadIdx.x & 31) & ~3;
        float p0 = __shfl_sync(0xFFFFFFFFu, p, qbase + 0), p1 = __shfl_sync(0xFFFFFFFFu, p, qbase + 1);
        float p2 = __shfl_sync(0xFFFFFFFFu, p, qbase + 2), p3 = __shfl_sync(0xFFFFFFFFu, p, qbase + 3);
        if (valid && j == 0 && args.action) {
            uint32_t a;
            if (args.greedy) {
                // int(np.argmax(probs * mask)): first maximum wins (reinforce_agent.py:179-185)
                float q0 = (fl & 1u) ? p0 : 0.0f, q1 = (fl & 2u) ? p1 : 0.0f, q2 = (fl & 4u) ? p2 : 0.0f,
                      q3 = (fl & 8u) ? p3 : 0.0f;
                if (!use_mask) { q0 = p0; q1 = p1; q2 = p2; q3 = p3; }
                a = 0; float best = q0;
                if (q1 > best) { best = q1; a = 1; }
                if (q2 > best) { best = q2; a = 2; }
                if (q3 > best) { best = q3; a = 3; }
            } else if constexpr (kNp) {
                b2048_np_rng r = npa.rng[s];
                a = np::choice4(r, p0, p1, p2, p3);   // rng.choice(4, p=probs) (reinforce_agent.py:187)
                npa.rng[s] = r;
            } else {
                // rng.choice(4, p=probs) == inverse CDF on one uniform (reinforce_agent.py:187); the uniform
                // is word 3 of the board's Philox block for this step
                Rand4 r = stream(args.seed, args.gid0 + (uint64_t)s, args.t, B2048_DOM_STEP);
                float c0 = p0, c1 = c0 + p1, c2 = c1 + p2, c3 = c2 + p3;
                float u = ((float)(r.w3 >> 8) + 0.5f) * (1.0f / 16777216.0f) * c3;
                a = (u >= c0 ? 1u : 0u) + (u >= c1 ? 1u : 0u) + (u >= c2 ? 1u : 0u);
                // never return a zero-probability (masked) action because of rounding at a CDF edge
                float pa = a == 0 ? p0 : a == 1 ? p1 : a == 2 ? p2 : p3;
                if (!(pa > 0.0f)) {
                    if (p3 > 0.0f) a = 3;
                    if (p2 > 0.0f) a = 2;
                    if (p1 > 0.0f) a = 1;
                    if (p0 > 0.0f) a = 0;
                }
            }
            args.action[s] = (uint8_t)a;
        }
        __syncthreads();  // arena is reused by the next tile
    }
}

__global__ void __launch_bounds__(kMlpThreads, 1) policy_step_kernel(const __grid_constant__ PolicyArgs args) {
    policy_step_body<false>(args, PolicyNpArgs{});
}

__global__ void __launch_bounds__(kMlpThreads, 1) policy_step_np_kernel(const __grid_constant__ PolicyArgs args,
                                                                         const __grid_constant__ PolicyNpArgs npa) {
    policy_step_body<true>(args, npa);
}

struct ForwardArgs {
    MlpDev mlp;
    const uint64_t* board;
    float* out;
    int64_t n;
};

__global__ void __launch_bounds__(kMlpThreads, 1) mlp_forward_kernel(const __grid_constant__ ForwardArgs args) {
    extern __shared__ __align__(16) float arena[];
    const MlpDev& m = args.mlp;
    const int n_out = m.dims[m.n_layers];
    const int64_t n_tiles = (args.n + kTileM - 1) / kTileM;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t s0 = tile * kTileM;
        tile_forward_hidden(arena, m, args.board, s0, args.n, nullptr);
        float v = tile_head(arena, m);
        const int b = threadIdx.x >> 2, j = threadIdx.x & 3;
        if (s0 + b < args.n && j < n_out) args.out[(s0 + b) * n_out + j] = v;
        __syncthreads();
    }
}

// forward_logits on explicit float32 input vectors (the reference's own signature, src/MLP.py:159-196):
// used by the drop-in MLP.forward_logits; returns logits and, optionally, every activation / pre-activation.
struct DenseArgs {
    MlpDev mlp;
    const float* x;
    float* act_out[B2048_MAX_LAYERS + 1];  // act_out[l+1] = a_{l+1} (act_out[L] = logits); may be NULL
    float* pre_out[B2048_MAX_LAYERS];      // pre_out[l] = z_l; may be NULL
    int64_t n;
    int buf_stride;
};

__global__ void __launch_bounds__(kMlpThreads, 1) dense_forward_kernel(const __grid_constant__ DenseArgs args) {
    extern __shared__ __align__(16) float arena[];
    const MlpDev& m = args.mlp;
    const int L = m.n_layers;
    const int bs = args.buf_stride;
    float* buf0 = arena;
    float* buf1 = arena + (size_t)kTileM * bs;
    const int64_t n_tiles = (args.n + kTileM - 1) / kTileM;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t s0 = tile * kTileM;
        const int in0 = m.dims[0];
        for (int idx = threadIdx.x; idx < kTileM * in0; idx += kMlpThreads) {
            int b = idx / in0, k = idx - b * in0;
            buf0[b * bs + k] = (s0 + b < args.n) ? args.x[(s0 + b) * in0 + k] : 0.0f;
        }
        __syncthreads();
        float* in = buf0;
        float* out = buf1;
        for (int l = 0; l < L; ++l) {
            tile_layer<0>(in, m.dims[l], bs, m.W[l], m.b[l], m.dims[l + 1], out, bs, m.activation, l + 1 < L,
                          args.act_out[l + 1], s0, args.n, args.pre_out[l]);
            __syncthreads();
            float* tmp = in; in = out; out = tmp;
        }
    }
}

int validate_mlp(const b2048_mlp_desc* d, MlpDev* out, size_t* smem_bytes, int smem_optin, const char* who) {
    if (!d) return fail(B2048_ERR_INVALID, std::string(who) + ": mlp descriptor is NULL");
    if (d->n_layers < 1 || d->n_layers > B2048_MAX_LAYERS)
        return fail(B2048_ERR_INVALID, std::string(who) + ": n_layers out of range");
    if (d->activation != B2048_ACTV_SIGMOID && d->activation != B2048_ACTV_RELU)
        return fail(B2048_ERR_INVALID, std::string(who) + ": unsupported activation");  // MLP.py:135-136
    if (d->obs_mode < B2048_OBS_RAW || d->obs_mode > B2048_OBS_ONEHOT)
        return fail(B2048_ERR_INVALID, std::string(who) + ": unsupported obs_mode");
    const int in0 = d->obs_mode == B2048_OBS_ONEHOT ? 272 : 16;
    if (d->dims[0] != in0) return fail(B2048_ERR_INVALID, std::string(who) + ": dims[0] must be 16 (raw/log2) or 272 (onehot)");
    const int n_out = d->dims[d->n_layers];
    if (n_out < 1 || n_out > 4) return fail(B2048_ERR_UNSUPPORTED, std::string(who) + ": 1..4 outputs supported");
    for (int l = 1; l < d->n_layers; ++l)
        if (d->dims[l] < 4 || d->dims[l] % 4 != 0 || d->dims[l] > 1024)
            return fail(B2048_ERR_UNSUPPORTED, std::string(who) + ": hidden sizes must be multiples of 4 in [4,1024]");
    for (int l = 0; l < d->n_layers; ++l)
        if (!d->W[l] || !d->b[l]) return fail(B2048_ERR_INVALID, std::string(who) + ": NULL parameter pointer");
    out->n_layers = d->n_layers; out->activation = d->activation; out->obs_mode = d->obs_mode;
    out->obs_scale = d->obs_log2_scale;
    for (int l = 0; l <= d->n_layers; ++l) out->dims[l] = d->dims[l];
    for (int l = 0; l < d->n_layers; ++l) { out->W[l] = d->W[l]; out->b[l] = d->b[l]; }
    *smem_bytes = mlp_arena_bytes(out->dims, out->n_layers);
    if (*smem_bytes > (size_t)smem_optin)
        return fail(B2048_ERR_UNSUPPORTED, std::string(who) + ": hidden layers too wide for the shared-memory activation arena");
    return B2048_OK;
}

}  // namespace b2

using namespace b2;

static int policy_step_impl(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags, const b2048_mlp_desc* mlp,
                            uint8_t* action, float* probs, float* logits, int64_t n, uint64_t seed, uint64_t gid0,
                            uint32_t t, int32_t greedy, int32_t precision, void* stream, bool rebuild_image);

extern "C" int b2048_policy_step(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags,
                                 const b2048_mlp_desc* mlp, uint8_t* action, float* probs, float* logits, int64_t n,
                                 uint64_t seed, uint64_t gid0, uint32_t t, int32_t greedy, int32_t precision,
                                 void* stream) {
    return policy_step_impl(h, board, mask_flags, mlp, action, probs, logits, n, seed, gid0, t, greedy, precision, stream,
                            true);
}

// Live-board list of a run-to-termination rollout: slot_map[0 .. *count) = the boards whose episode is still running
// (ep_len[b] == 0), in no particular order (a board's results do not depend on its slot).  *count must be zero on entry.
__global__ void __launch_bounds__(256) compact_live_kernel(const int32_t* __restrict__ ep_len, int64_t B,
                                                            int32_t* __restrict__ slot_map, int32_t* __restrict__ count) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool live = b < B && ep_len[b] == 0;
    const uint32_t m = __ballot_sync(0xFFFFFFFFu, live);
    if (m == 0u) return;
    const int lane = threadIdx.x & 31, leader = __ffs((int)m) - 1;
    int base = 0;
    if (lane == leader) base = atomicAdd(count, __popc(m));
    base = __shfl_sync(0xFFFFFFFFu, base, leader);
    if (live) slot_map[base + __popc(m & ((1u << lane) - 1u))] = (int32_t)b;
}

extern "C" int b2048_compact_live(b2048_handle* h, const int32_t* ep_len, int64_t B, int32_t* slot_map, int32_t* count,
                                  void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_compact_live: handle is NULL");
    B2_REQUIRE(B >= 0 && B < ((int64_t)1 << 31), "b2048_compact_live: B out of range");
    B2_REQUIRE(ep_len && slot_map && count, "b2048_compact_live: NULL buffer");
    cudaStream_t s = (cudaStream_t)stream;
    B2_CUDA(cudaMemsetAsync(count, 0, sizeof(int32_t), s));
    if (B == 0) return B2048_OK;
    compact_live_kernel<<<(unsigned)((B + 255) / 256), 256, 0, s>>>(ep_len, B, slot_map, count);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

// The rollout loop of ReinforceAgent.run_episode (reference src/reinforce_agent.py:221-236) for a whole batch, issued
// from C so that a rollout step costs two kernel launches and no interpreter time: for k in [0, n_steps):
//   t = t_begin + k;  actions[t] = policy(boards[t], flags[t]);  (boards[t+1], flags[t+1], rewards[t]) = step(...)
extern "C" int b2048_rollout_many(b2048_handle* h, uint64_t* boards, uint8_t* flags, uint8_t* actions, float* rewards,
                                  uint32_t* score, uint32_t* step, uint8_t* max_exp, int32_t* ep_len,
                                  const b2048_env_cfg* cfg, const b2048_mlp_desc* mlp, int64_t B, int32_t t_begin,
                                  int32_t n_steps, uint64_t seed, uint64_t gid0, uint32_t t0, int32_t use_mask,
                                  int32_t greedy, int32_t precision, const int32_t* slot_map, int64_t n_slots,
                                  const int32_t* n_slots_dev, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_rollout_many: handle is NULL");
    B2_REQUIRE(B >= 0 && n_steps >= 0 && t_begin >= 0, "b2048_rollout_many: negative size");
    if (B == 0 || n_steps == 0) return B2048_OK;
    B2_REQUIRE(boards && flags && actions && rewards && cfg && mlp, "b2048_rollout_many: NULL buffer");
    b2048_env_cfg c = *cfg;
    c.action_mode = B2048_ACT_BUFFER;
    if (precision == 1) {
        // one persistent launch for the whole horizon (policy on tcgen05 + env step in the same kernel)
        int st = launch_rollout_tc(h, mlp, boards, flags, actions, rewards, score, step, max_exp, ep_len, &c, B, t_begin, n_steps,
                                   seed, gid0, t0, use_mask, greedy, slot_map, n_slots, n_slots_dev, (cudaStream_t)stream);
        if (st != B2048_ERR_UNSUPPORTED) return st;
    }
    // Shapes of the shape-generic tensor-core policy kernel: the POLICY step visits only the listed boards; the step kernel
    // passes finished boards through untouched anyway (ep_len != 0).
    const bool gen_slots = slot_map != nullptr;
    if (gen_slots) {
        B2_REQUIRE(precision == 1 && gen_supported(h, mlp) && ep_len != nullptr && n_slots >= 0 && n_slots <= B,
                   "b2048_rollout_many: slot_map needs a tensor-core policy (precision 1; the fused 16-256-256-4 rollout kernel with "
                   "an action-mask-on env configuration and B >= 4096, or a shape of the generic tcgen05 policy kernel) and ep_len");
        if (n_slots == 0) return B2048_OK;
    }
    for (int32_t k = 0; k < n_steps; ++k) {
        const int64_t t = (int64_t)t_begin + k;
        const uint32_t t_env = t0 + (uint32_t)t + 1u;
        uint64_t* b_in = boards + t * B;
        uint8_t* f_in = flags + t * B;
        int st = gen_slots ? launch_forward_gen(h, mlp, b_in, use_mask ? f_in : nullptr, nullptr, actions + t * B, nullptr, nullptr,
                                                n_slots, seed, gid0, t_env, greedy, 0, k == 0, (cudaStream_t)stream, slot_map, n_slots_dev)
                           : policy_step_impl(h, b_in, use_mask ? f_in : nullptr, mlp, actions + t * B, nullptr, nullptr, B, seed, gid0,
                                              t_env, greedy, precision, stream, k == 0);
        if (st != B2048_OK) return st;
        st = b2048_step_many(h, b_in, b_in + B, score, step, max_exp, actions + t * B, nullptr, f_in, nullptr, &c, nullptr,
                             rewards + t * B, nullptr, f_in + B, nullptr, ep_len, (uint32_t)(t + 1), B, seed, gid0, t_env,
                             stream);
        if (st != B2048_OK) return st;
    }
    return B2048_OK;
}

// b2048_rollout_many's run-to-termination loop with the reference's NumPy streams: policy_step_np_kernel (fp32) over the
// listed boards, then the generic step kernel's NumPy variant over all B (it passes the finished boards through).
extern "C" int b2048_rollout_many_np(b2048_handle* h, uint64_t* boards, uint8_t* flags, uint8_t* actions, float* rewards,
                                     uint32_t* score, uint32_t* step, uint8_t* max_exp, int32_t* ep_len,
                                     const b2048_env_cfg* cfg, const b2048_mlp_desc* mlp, int64_t B, int32_t t_begin,
                                     int32_t n_steps, b2048_np_rng* env_rng, b2048_np_rng* policy_rng, int32_t use_mask,
                                     int32_t greedy, const int32_t* slot_map, int64_t n_slots, const int32_t* n_slots_dev,
                                     void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_rollout_many_np: handle is NULL");
    B2_REQUIRE(B >= 0 && n_steps >= 0 && t_begin >= 0, "b2048_rollout_many_np: negative size");
    if (B == 0 || n_steps == 0) return B2048_OK;
    B2_REQUIRE(boards && flags && actions && rewards && cfg && mlp && ep_len && env_rng && policy_rng,
               "b2048_rollout_many_np: NULL buffer (ep_len, env_rng and policy_rng are required)");
    B2_REQUIRE(!cfg->auto_reset, "b2048_rollout_many_np: run-to-termination only (cfg->auto_reset must be 0)");
    B2_REQUIRE(cfg->reward_mode == B2048_REWARD_SUM || cfg->reward_mode == B2048_REWARD_LOG2,
               "b2048_rollout_many_np: unsupported reward mode");
    B2_REQUIRE(cfg->bonus_mode >= B2048_BONUS_OFF && cfg->bonus_mode <= B2048_BONUS_LOG2,
               "b2048_rollout_many_np: unsupported bonus mode");
    B2_REQUIRE(slot_map == nullptr || (n_slots >= 0 && n_slots <= B), "b2048_rollout_many_np: n_slots out of range");
    b2048_env_cfg c = *cfg;
    c.action_mode = B2048_ACT_BUFFER;
    c.obs_mode = B2048_OBS_NONE;
    PolicyArgs a;
    size_t smem = 0;
    int st = validate_mlp(mlp, &a.mlp, &smem, h->smem_optin, "b2048_rollout_many_np");
    if (st != B2048_OK) return st;
    const int64_t n_pol = slot_map ? n_slots : B;
    if (n_pol == 0) return B2048_OK;
    B2_CUDA(cudaFuncSetAttribute(policy_step_np_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int64_t tiles = (n_pol + kTileM - 1) / kTileM;
    const int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
    cudaStream_t s = (cudaStream_t)stream;
    PolicyNpArgs npa;
    npa.rng = policy_rng; npa.ep_len = ep_len; npa.slot_map = slot_map; npa.n_dev = slot_map ? n_slots_dev : nullptr;
    a.probs = nullptr; a.logits = nullptr; a.n = n_pol; a.seed = 0; a.gid0 = 0; a.t = 0; a.greedy = greedy;
    for (int32_t k = 0; k < n_steps; ++k) {
        const int64_t t = (int64_t)t_begin + k;
        uint64_t* b_in = boards + t * B;
        uint8_t* f_in = flags + t * B;
        a.board = b_in; a.mask_flags = use_mask ? f_in : nullptr; a.action = actions + t * B;
        policy_step_np_kernel<<<grid, kMlpThreads, smem, s>>>(a, npa);
        B2_CUDA(cudaGetLastError());
        st = launch_step_np(h, b_in, b_in + B, score, step, max_exp, actions + t * B, f_in, &c, rewards + t * B, f_in + B, ep_len,
                            (uint32_t)(t + 1), B, env_rng, s);
        if (st != B2048_OK) return st;
    }
    return B2048_OK;
}

static int policy_step_impl(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags, const b2048_mlp_desc* mlp,
                            uint8_t* action, float* probs, float* logits, int64_t n, uint64_t seed, uint64_t gid0,
                            uint32_t t, int32_t greedy, int32_t precision, void* stream, bool rebuild_image) {
    B2_REQUIRE(h != nullptr, "b2048_policy_step: handle is NULL");
    B2_REQUIRE(n >= 0, "b2048_policy_step: n < 0");
    if (n == 0) return B2048_OK;
    B2_REQUIRE(board != nullptr, "b2048_policy_step: board is NULL");
    PolicyArgs a;
    size_t smem = 0;
    int st = validate_mlp(mlp, &a.mlp, &smem, h->smem_optin, "b2048_policy_step");
    if (st != B2048_OK) return st;
    if (precision == 1) {
        st = launch_policy_tc(h, mlp, board, mask_flags, action, probs, logits, n, seed, gid0, t, greedy, (cudaStream_t)stream,
                              rebuild_image);
        if (st == B2048_ERR_UNSUPPORTED)      // other shapes: the shape-generic kernel, one fp16 MMA per product
            st = launch_forward_gen(h, mlp, board, mask_flags, nullptr, action, probs, logits, n, seed, gid0, t, greedy, 0,
                                    rebuild_image, (cudaStream_t)stream);
        if (st == B2048_ERR_UNSUPPORTED)
            return fail(B2048_ERR_UNSUPPORTED,
                        "b2048_policy_step: precision 1 (tcgen05) implements ReLU policies with 1-4 hidden layers of 64 / 128 / 192 / "
                        "256 units on log2 / one-hot observations (16-256-256-4 also on raw ones), n >= 4096; use precision 0");
        return st;
    }
    if (precision != 0) return fail(B2048_ERR_INVALID, "b2048_policy_step: precision must be 0 (fp32) or 1 (bf16 tcgen05)");
    a.board = board; a.mask_flags = mask_flags; a.action = action; a.probs = probs; a.logits = logits;
    a.n = n; a.seed = seed; a.gid0 = gid0; a.t = t; a.greedy = greedy;
    B2_CUDA(cudaFuncSetAttribute(policy_step_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t tiles = (n + kTileM - 1) / kTileM;
    int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
    policy_step_kernel<<<grid, kMlpThreads, smem, (cudaStream_t)stream>>>(a);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_mlp_forward(b2048_handle* h, const uint64_t* board, const b2048_mlp_desc* mlp, float* out,
                                 int64_t n, int32_t precision, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_mlp_forward: handle is NULL");
    B2_REQUIRE(n >= 0, "b2048_mlp_forward: n < 0");
    if (n == 0) return B2048_OK;
    B2_REQUIRE(board != nullptr && out != nullptr && mlp != nullptr, "b2048_mlp_forward: board/out/mlp is NULL");
    B2_REQUIRE(precision >= 0 && precision <= 3,
               "b2048_mlp_forward: precision must be 0 (fp32), 1 (bf16 tcgen05), 2 (auto) or 3 (split-fp16 tcgen05)");
    if (precision == 2 || precision == 3) {   // float32-grade tensor-core forward (what "auto" selects)
        int st = launch_forward_hp(h, mlp, board, out, n, (cudaStream_t)stream);
        if (st == B2048_ERR_UNSUPPORTED)
            st = launch_forward_gen(h, mlp, board, nullptr, out, nullptr, nullptr, nullptr, n, 0, 0, 0, 1, 1, true, (cudaStream_t)stream);
        if (st != B2048_ERR_UNSUPPORTED) return st;
        if (precision == 3)
            return fail(B2048_ERR_UNSUPPORTED,
                        "b2048_mlp_forward: precision 3 (split-fp16 tcgen05) implements ReLU networks with 1-4 hidden layers of 64 / 128 / "
                        "192 / 256 units on log2 / one-hot observations with n >= 4096 only");
    }
    if (precision == 1) {
        int st = launch_forward_tc(h, mlp, board, out, n, (cudaStream_t)stream);
        if (st == B2048_ERR_UNSUPPORTED)
            st = launch_forward_gen(h, mlp, board, nullptr, out, nullptr, nullptr, nullptr, n, 0, 0, 0, 1, 0, true, (cudaStream_t)stream);
        if (st != B2048_ERR_UNSUPPORTED) return st;
        return fail(B2048_ERR_UNSUPPORTED,
                    "b2048_mlp_forward: precision 1 (bf16 tcgen05) implements 16-256-256-(<=4) ReLU networks on raw/log2 "
                    "observations with n >= 4096 only");
    }
    ForwardArgs a;
    size_t smem = 0;
    int st = validate_mlp(mlp, &a.mlp, &smem, h->smem_optin, "b2048_mlp_forward");
    if (st != B2048_OK) return st;
    a.board = board; a.out = out; a.n = n;
    B2_CUDA(cudaFuncSetAttribute(mlp_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t tiles = (n + kTileM - 1) / kTileM;
    int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
    mlp_forward_kernel<<<grid, kMlpThreads, smem, (cudaStream_t)stream>>>(a);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}

extern "C" int b2048_dense_forward(b2048_handle* h, const float* x, const b2048_mlp_desc* mlp, float* const* act_out,
                                   float* const* pre_out, int64_t n, void* stream) {
    B2_REQUIRE(h != nullptr, "b2048_dense_forward: handle is NULL");
    B2_REQUIRE(n >= 0, "b2048_dense_forward: n < 0");
    if (n == 0) return B2048_OK;
    B2_REQUIRE(x != nullptr && mlp != nullptr, "b2048_dense_forward: x/mlp is NULL");
    B2_REQUIRE(mlp->n_layers >= 1 && mlp->n_layers <= B2048_MAX_LAYERS, "b2048_dense_forward: n_layers out of range");
    B2_REQUIRE(mlp->activation == B2048_ACTV_SIGMOID || mlp->activation == B2048_ACTV_RELU,
               "b2048_dense_forward: unsupported activation");
    DenseArgs a;
    int maxd = 0;
    for (int l = 0; l <= mlp->n_layers; ++l) {
        a.mlp.dims[l] = mlp->dims[l];
        if (mlp->dims[l] > maxd) maxd = mlp->dims[l];
        if (l < mlp->n_layers && (mlp->dims[l] < 4 || mlp->dims[l] % 4 != 0))
            return fail(B2048_ERR_UNSUPPORTED, "b2048_dense_forward: layer input widths must be multiples of 4");
    }
    a.mlp.n_layers = mlp->n_layers; a.mlp.activation = mlp->activation; a.mlp.obs_mode = mlp->obs_mode;
    a.mlp.obs_scale = mlp->obs_log2_scale;
    for (int l = 0; l < mlp->n_layers; ++l) {
        B2_REQUIRE(mlp->W[l] && mlp->b[l], "b2048_dense_forward: NULL parameter pointer");
        a.mlp.W[l] = mlp->W[l]; a.mlp.b[l] = mlp->b[l];
        a.pre_out[l] = pre_out ? pre_out[l] : nullptr;
    }
    for (int l = 0; l <= mlp->n_layers; ++l) a.act_out[l] = act_out ? act_out[l] : nullptr;
    a.x = x; a.n = n; a.buf_stride = ((maxd + 3) / 4) * 4 + kPad;
    size_t smem = (size_t)2 * kTileM * a.buf_stride * sizeof(float);
    if (smem > (size_t)h->smem_optin) return fail(B2048_ERR_UNSUPPORTED, "b2048_dense_forward: layers too wide");
    B2_CUDA(cudaFuncSetAttribute(dense_forward_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int64_t tiles = (n + kTileM - 1) / kTileM;
    int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
    dense_forward_kernel<<<grid, kMlpThreads, smem, (cudaStream_t)stream>>>(a);
    B2_CUDA(cudaGetLastError());
    return B2048_OK;
}
