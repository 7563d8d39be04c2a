// b2048_internal.h — things shared by the .cu translation units of libb2048 (not part of the ABI).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>

#include "../../include/b2048.h"

struct b2048_handle {
    uint8_t* d_tables;   // [131072 B lut_left (u16 x 65536)] [65536 B lut_merge (u8 x 65536)] [small tables]
    int device;
    int num_sms;
    int smem_optin;      // max opt-in dynamic shared memory per block
    uint8_t* tc_image;   // bf16 weight image of the tensor-core policy kernel (lazily allocated)
    uint8_t* hp_image;   // split-fp16 weight image of the float32-grade forward kernel (lazily allocated)
    uint8_t* gen_image;  // weight images of the shape-generic tensor-core kernels (b2048_mlp_gen.cu; lazily allocated)
    size_t gen_image_bytes;
    unsigned pipe_split; // B2048_DBG_PARAM_PIPE_SPLIT: CTAs per role of the update pipeline (0 = default split)
    unsigned debug;      // bit B2048_DBG_* set through b2048_debug_set (test / profiling switches; 0 in production)
    unsigned attrs;      // b2::Attr bits: the opt-in shared-memory attribute of that kernel family has been set on THIS device
                         // (cudaFuncSetAttribute is per device; a process may hold handles on several)
    long long* dbg_clock;   // in-kernel clocks (B2048_DBG_TC_CLOCKS / _STEP_CLOCKS), b2::DBG_CLOCK_SLOTS, on this device
    int* dbg_progress;      // mapped pinned host block: the update pipeline's progress words (B2048_DBG_TC_CLOCKS)
};

#define B2048_LUT_LEFT_BYTES 131072
#define B2048_LUT_MERGE_BYTES 65536
#define B2048_LUT_BYTES (B2048_LUT_LEFT_BYTES + B2048_LUT_MERGE_BYTES)
// the small tables of b2048_step_fast.cuh follow the row tables in the same allocation
#define B2048_TABLES_BYTES (B2048_LUT_BYTES + 2048 + 128 + 64)

namespace b2 {

void set_error(const std::string& msg);
int fail(b2048_status st, const std::string& msg);
int check_cuda(cudaError_t e, const char* what);

inline const uint16_t* lut_left_ptr(const b2048_handle* h) { return reinterpret_cast<const uint16_t*>(h->d_tables); }
inline const uint8_t* lut_merge_ptr(const b2048_handle* h) { return h->d_tables + B2048_LUT_LEFT_BYTES; }

// Kernel families whose opt-in dynamic shared-memory size is set once per handle (bits of b2048_handle::attrs).
enum Attr : unsigned {
    ATTR_POLICY_TC = 1u,   // policy_tc_kernel (policy, forward, fused rollout)
    ATTR_FB_TC = 2u,       // fb_tc_kernel
    ATTR_ATB_256 = 4u,     // atb_tc_kernel<256>
    ATTR_ATB_16 = 8u,      // atb_tc_kernel<16>
    ATTR_HP = 16u,         // fwd_hp_kernel, bwd_tc_kernel, update_pipe_kernel
    ATTR_GEN = 32u,        // gen_mlp_kernel, gen_dw_kernel
};

// ---- which tensor-core family takes a network
// The hand-specialised network of the fixed-shape kernels: 16 -> 256 -> 256 -> anything.
inline bool is_16_256_256(const b2048_mlp_desc* m) {
    return m->n_layers == 3 && m->dims[0] == 16 && m->dims[1] == 256 && m->dims[2] == 256;
}
// ... as those kernels implement it: ReLU, 1..4 outputs, raw or log2 observations.  Each launcher adds its own limits.
inline bool fixed_tc_net(const b2048_mlp_desc* m) {
    return is_16_256_256(m) && m->dims[3] >= 1 && m->dims[3] <= 4 && m->activation == B2048_ACTV_RELU &&
           (m->obs_mode == B2048_OBS_RAW || m->obs_mode == B2048_OBS_LOG2);
}
// The shapes of the shape-generic kernels (b2048_mlp_gen.cu); gen_supported() also checks the device.
bool gen_shape_ok(const b2048_mlp_desc* mlp);
bool gen_supported(const b2048_handle* h, const b2048_mlp_desc* mlp);

// Pointers of the per-layer weight and bias gradients inside the flat gradient vector (layout W_0, b_0, W_1, b_1, ...).
inline void carve_grads(const b2048_mlp_desc* mlp, float* grads, float** gW, float** gb) {
    for (int l = 0; l < mlp->n_layers; ++l) {
        gW[l] = grads; grads += (int64_t)mlp->dims[l] * mlp->dims[l + 1];
        gb[l] = grads; grads += mlp->dims[l + 1];
    }
}

// ---- in-kernel clocks (B2048_DBG_TC_CLOCKS, B2048_DBG_STEP_CLOCKS); b2048_debug_set allocates the handle's buffers
constexpr int DBG_CLOCK_SLOTS = 256;        // the most any instrumented kernel records
constexpr int DBG_PROGRESS_WORDS = 256 * 8; // update pipeline: 8 words per CTA
// The handle's clock buffer, zeroed on `stream`, if debug option `option` is set; else nullptr.
long long* debug_clock_begin(const b2048_handle* h, int option, cudaStream_t stream);
// Waits for `stream`, then copies the first `count` slots of the clock buffer to `host`.
int debug_clock_read(const b2048_handle* h, long long* host, int count, cudaStream_t stream);

// ---- b2048_policy.cu
struct MlpDev;
int validate_mlp(const b2048_mlp_desc* d, MlpDev* out, size_t* smem_bytes, int smem_optin, const char* who);

// ---- b2048_policy_tc.cu: the bf16 kernels of the 16-256-256 network.  The launchers return B2048_ERR_UNSUPPORTED
// (without an error message) for a network or size they do not implement.
int ensure_tc_image(b2048_handle* h);
void launch_tc_prepare(const b2048_mlp_desc* mlp, uint8_t* img, cudaStream_t stream);
int launch_policy_tc(b2048_handle* h, const b2048_mlp_desc* mlp, const uint64_t* board, const uint8_t* mask_flags,
                     uint8_t* action, float* probs, float* logits, int64_t n, uint64_t seed, uint64_t gid0, uint32_t t,
                     int greedy, cudaStream_t stream, bool rebuild_image);
int launch_forward_tc(b2048_handle* h, const b2048_mlp_desc* mlp, const uint64_t* board, float* out, int64_t n,
                      cudaStream_t stream);
int launch_rollout_tc(b2048_handle* h, const b2048_mlp_desc* mlp, uint64_t* boards, uint8_t* flags, uint8_t* actions,
                      float* rewards, uint32_t* score, uint32_t* step, uint8_t* max_exp, int32_t* ep_len,
                      const b2048_env_cfg* cfg, int64_t B, int32_t t_begin, int32_t n_steps, uint64_t seed, uint64_t gid0,
                      uint32_t t0, int use_mask, int greedy, const int32_t* slot_map, int64_t n_slots, const int32_t* n_slots_dev,
                      cudaStream_t stream);

// ---- b2048_learn_tc.cu: single-bf16 gradients of the 16-256-256 network
bool backward_tc_supported(const b2048_handle* h, const b2048_mlp_desc* mlp);
int64_t backward_tc_workspace_bytes(int64_t chunk);
int launch_backward_tc(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags, const uint8_t* action,
                       const float* coef, const b2048_mlp_desc* mlp, float* grads, int64_t n, int head_mode,
                       uint8_t* workspace, int64_t chunk, cudaStream_t stream);

// ---- b2048_learn_hp.cu: float32-grade (split-fp16) forward and gradients of the 16-256-256 network
bool backward_hp_supported(const b2048_handle* h, const b2048_mlp_desc* mlp);
int64_t backward_hp_workspace_bytes(int64_t chunk);
int launch_forward_hp(b2048_handle* h, const b2048_mlp_desc* mlp, const uint64_t* board, float* out, int64_t n, cudaStream_t stream);
int launch_backward_hp(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags, const uint8_t* action,
                       const float* coef, const b2048_mlp_desc* mlp, float* grads, int64_t n, int head_mode,
                       uint8_t* workspace, int64_t workspace_bytes, int64_t chunk, cudaStream_t stream,
                       const float* ent_coef = nullptr, double* ent_sum = nullptr);
// scale[0] = S, the power of two that brings max |coef[0 .. n)| into [32, 64); scale[1] = 1 / S; scale[2] = bits of the max.
// The fp16 backward passes multiply their deltas by S.  ent_coef != NULL (the entropy bonus): the max is taken of
// |coef| + 1.5 |ent_coef|, a bound of the head delta (b2048_entropy.cuh).
int launch_loss_scale(const b2048_handle* h, const float* coef, int64_t n, float* scale, cudaStream_t stream,
                      const float* ent_coef = nullptr);

// ---- b2048_mlp_gen.cu: the shape-generic kernels
int64_t gen_workspace_bytes(const b2048_mlp_desc* mlp, int64_t chunk);
int launch_forward_gen(b2048_handle* h, const b2048_mlp_desc* mlp, const uint64_t* board, const uint8_t* mask_flags, float* out,
                       uint8_t* action, float* probs, float* logits, int64_t n, uint64_t seed, uint64_t gid0, uint32_t t, int greedy,
                       int split, bool rebuild_image, cudaStream_t stream, const int32_t* slot_map = nullptr,
                       const int32_t* n_dev = nullptr);
int launch_backward_gen(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags, const uint8_t* action, const float* coef,
                        const b2048_mlp_desc* mlp, float* grads, int64_t n, int head_mode, uint8_t* workspace, int64_t chunk,
                        cudaStream_t stream, const float* ent_coef = nullptr, double* ent_sum = nullptr);

// ---- b2048_env.cu: the step of b2048_rollout_many_np (generic step kernel, spawns from the boards' NumPy env streams)
int launch_step_np(b2048_handle* h, const uint64_t* board_in, uint64_t* board_out, uint32_t* score, uint32_t* step,
                   uint8_t* max_exp, const uint8_t* action, const uint8_t* flags_in, const b2048_env_cfg* cfg, float* reward,
                   uint8_t* flags, int32_t* ep_len, uint32_t ep_t, int64_t n, b2048_np_rng* env_rng, cudaStream_t s);

}  // namespace b2

#define B2_CUDA(expr)                                              \
    do {                                                           \
        int _st = b2::check_cuda((expr), #expr);                   \
        if (_st != B2048_OK) return _st;                           \
    } while (0)

#define B2_REQUIRE(cond, msg)                                      \
    do {                                                           \
        if (!(cond)) return b2::fail(B2048_ERR_INVALID, msg);      \
    } while (0)
