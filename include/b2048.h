/*
 * b2048.h — C ABI of libb2048: the B200-native batched 2048 environment and
 * rollout engine (hand-written sm_100a CUDA behind plain C entry points).
 *
 * Drop-in boundary.  The reference (pqpeqr/RL-2048-with-Reinforce-and-Actor-Critic)
 * is pure Python: its seam is the class API in src/game2048.py, src/env.py,
 * src/MLP.py and src/reinforce_agent.py.  Every entry point below names the
 * reference function(s) (file:line) whose arithmetic it replaces; the Python
 * host mirror in rl-2048-with-reinforce-and-actor-critic_b200/ binds these
 * symbols with ctypes and re-exposes the reference's own class API.
 *
 * Contract (all entry points):
 *   - plain C types only; no C++ / torch types cross the boundary;
 *   - every buffer pointer is a DEVICE pointer owned by the caller unless a
 *     parameter is documented as "host"; the library never frees caller memory;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default
 *     stream); every call is asynchronous with respect to the host;
 *   - return value: 0 = B2048_OK, otherwise a b2048_status; the message of the
 *     last failure on the calling thread is returned by b2048_last_error();
 *   - the device is whatever is current (cudaSetDevice) on the calling thread;
 *     one process per GPU under multi-GPU.
 *
 * Packed board: one uint64 per board, sixteen 4-bit exponents; cell (r, c) of
 * Game2048.board (game2048.py:16) lives in bits [4*(4r+c), 4*(4r+c)+4); 0 means
 * empty, e means tile 2^e (e <= 15, i.e. tiles up to 32768).  A 15+15 merge is
 * outside the domain and raises B2048_F_OVERFLOW for that board.
 *
 * Random streams: Philox4x32-10, key = (seed_lo, seed_hi),
 * counter = (gid_lo, gid_hi, t, domain) with gid the GLOBAL board id
 * (gid0 + index) and t the caller's global step index — so results do not
 * depend on how boards are sharded over ranks.
 *   domain B2048_DOM_STEP : w0 spawn cell, w1 spawn value, w2 env-side random
 *                           action, w3 policy-sampling uniform
 *   domain B2048_DOM_RESET: (w0, w1) first spawn, (w2, w3) second spawn
 * spawn(wp, wv): n = #empty; n == 0 -> no-op; k = mulhi32(wp, n); the k-th
 * empty cell in row-major order (np.argwhere order, game2048.py:109) receives
 * exponent 2 if wv >= 0xE6666667 (u = wv/2^32 >= 0.9, game2048.py:117) else 1.
 * The reference's own NumPy streams (default_rng(env_seed) / default_rng(policy_seed)) are a second, per-board
 * family: see b2048_np_rng below.
 */
#ifndef B2048_H_
#define B2048_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    B2048_OK = 0,
    B2048_ERR_INVALID = 1,   /* bad argument (NULL pointer, bad mode, n < 0, size != 4 ...) */
    B2048_ERR_CUDA = 2,      /* a CUDA runtime call failed */
    B2048_ERR_UNSUPPORTED = 3/* configuration outside what the kernels implement */
} b2048_status;

/* flags byte written per board by reset_many / step_many */
#define B2048_F_MASK      0x0Fu  /* bit a: action a is legal on the RETURNED board (0 up,1 right,2 down,3 left; game2048.py:9,95-99) */
#define B2048_F_CHANGED   0x10u  /* the move changed the board (is_changed, game2048.py:50) */
#define B2048_F_DONE      0x20u  /* terminated (game2048.py:172-187 after the spawn) */
#define B2048_F_TRUNC     0x40u  /* truncated (env.py:279-286) */
#define B2048_F_OVERFLOW  0x80u  /* a 32768+32768 merge happened: board left the 4-bit domain */

#define B2048_DOM_STEP  0u
#define B2048_DOM_RESET 1u

enum { B2048_REWARD_SUM = 0, B2048_REWARD_LOG2 = 1 };            /* env.py:212-223 */
enum { B2048_BONUS_OFF = 0, B2048_BONUS_RAW = 1, B2048_BONUS_LOG2 = 2 }; /* env.py:242-249 */
enum { B2048_OBS_NONE = 0, B2048_OBS_RAW = 1, B2048_OBS_LOG2 = 2, B2048_OBS_ONEHOT = 3 }; /* env.py:131-150 */
enum { B2048_ACT_BUFFER = 0,      /* actions read from the `action` buffer */
       B2048_ACT_RANDOM_LEGAL = 1,/* uniform over the legal mask (tools/simple_action_gen.py:7-13) from Philox w2 */
       B2048_ACT_RANDOM_ANY = 2,  /* uniform over {0,1,2,3}, illegal moves included */
       B2048_ACT_PRIORITY = 3     /* first LEGAL action in the fixed order cfg.action_priority (nibble k = k-th
                                     choice): tools/simple_action_gen.py:16-33, 0x3210 = up,right,down,left
                                     (action_gen_1), 0x2310 = up,right,left,down (action_gen_2); 0 if none is legal */ };

/* Mirrors Game2048EnvConfig (env.py:19-40); doubles because the reference
 * combines the reward in Python float64 (env.py:197-261). */
typedef struct b2048_env_cfg {
    int32_t reward_mode;            /* B2048_REWARD_*   */
    int32_t bonus_mode;             /* B2048_BONUS_*    */
    int32_t obs_mode;               /* B2048_OBS_*      */
    int32_t use_action_mask;        /* env.py:38        */
    int32_t max_steps;              /* env.py:40; <= 0 means None (never truncate) */
    int32_t action_mode;            /* B2048_ACT_*      */
    int32_t auto_reset;             /* 1: a board that terminated/truncated is reset in the same call */
    int32_t action_priority;        /* B2048_ACT_PRIORITY only (else 0) */
    double base_reward_scale;       /* env.py:27 */
    double empty_tile_reward;       /* env.py:29 */
    double merge_reward;            /* env.py:30 */
    double bonus_scale;             /* env.py:33 */
    double step_reward;             /* env.py:35 */
    double endgame_penalty;         /* env.py:36 */
    double invalid_action_penalty;  /* env.py:39 */
    float  obs_log2_scale;          /* env.py:24 (applied in float32 like numpy does) */
    float  reserved_f;
} b2048_env_cfg;

typedef struct b2048_handle b2048_handle;

/* Library-owned object holding the 65,536-entry row-transition tables
 * (Game2048._row_move_left, game2048.py:120-137, tabulated on the device). */
int b2048_create(b2048_handle** out);
int b2048_destroy(b2048_handle* h);
const char* b2048_last_error(void);
int b2048_version(void);

/* Test / profiling switches of one handle (all off by default; production code never sets them).  They replace
 * process-wide environment variables: the parity tests use them to reach the non-fused fall-back kernels so that
 * the fused ones can be compared with them bit for bit. */
enum { B2048_DBG_NO_FUSED_ROLLOUT = 0, /* b2048_rollout_many: always the policy-kernel / step-kernel loop */
       B2048_DBG_NO_FAST_STEP = 1,     /* b2048_step_many: always the generic step_kernel */
       B2048_DBG_TC_CLOCKS = 2,        /* tensor-core kernels record in-kernel phase clocks and print them to stderr */
       B2048_DBG_STEP_CLOCKS = 3,      /* the fast step kernel records per-iteration clocks and prints them to stderr */
       B2048_DBG_NO_PDL = 4,           /* launch without programmatic dependent launch (plain stream order) */
       B2048_DBG_NO_UPDATE_PIPE = 5,   /* b2048_mlp_backward precision 3: always the chunked kernel sequence, never the persistent pipeline */
       B2048_DBG_COUNT = 6,
       B2048_DBG_PARAM_PIPE_SPLIT = 16 /* integer parameter, not a flag: CTAs per role of the persistent update pipeline,
                                          value = backward | dW2 << 8 | dW1/dW3 << 16 (a zero field = default share) */ };
int b2048_debug_set(b2048_handle* h, int32_t option, int32_t value);

/* Copies the device tables back (host pointers; either may be NULL):
 * lut_left[65536]  : row after a left move (4 nibbles);
 * lut_merge[65536] : two nibbles = exponents of the (<= 2) merged tiles,
 *                    0 = none, 1 = the out-of-domain 15+15 merge (exponent 16). */
int b2048_get_row_lut(b2048_handle* h, uint16_t* lut_left_host, uint8_t* lut_merge_host);

/* Game2048.reset + Game2048Env.reset (game2048.py:26-34, env.py:174-194) for n boards.
 * score/step/max_exp may be NULL.  flags (may be NULL) receives the legal mask. */
int b2048_reset_many(b2048_handle* h, uint64_t* board, uint32_t* score, uint32_t* step,
                     uint8_t* max_exp, uint8_t* flags, const uint8_t* spawn_replay /* [n,2] or NULL */,
                     int64_t n, uint64_t seed, uint64_t gid0, uint32_t t, void* stream);

/* One fused environment step for n boards: Game2048.step/_move/_spawn/_is_done/
 * get_action_mask (game2048.py:40-70, :95-99, :108-187) + Game2048Env.step/
 * _compute_reward/_preprocess_board (env.py:131-150, :197-302).
 *   board_in / board_out : may alias (in-place) or be consecutive slices of a rollout buffer
 *   score, step, max_exp : per-board env state, updated in place; each may be NULL
 *                          (step == NULL disables truncation; max_exp == NULL disables the bonus)
 *   action               : uint8 per board, required for B2048_ACT_BUFFER (values taken & 3)
 *   action_out           : optional; receives the action actually played (useful for random modes)
 *   flags_in             : optional legal mask of board_in from the previous call (random-legal mode
 *                          reads it instead of recomputing); NULL -> recomputed
 *   spawn_replay         : optional uint8 per board; when bit 7 is set the spawn is NOT drawn from Philox
 *                          but replayed: bits 0-3 = index k of the empty cell (row-major), bit 4 = tile is a 4.
 *                          This is how the single-env drop-in reproduces the reference's NumPy-seeded games
 *                          (rng.integers / rng.random of game2048.py:113,117 are drawn by the host wrapper).
 *   merge_sum            : optional int32, sum of merged tiles (game2048.py:167-170)
 *   reward / reward64    : optional float32 / float64 reward (the float32 is the rounded float64)
 *   flags                : required uint8, B2048_F_*
 *   obs                  : optional float32 [n,16] (raw/log2) or [n,16,17] (onehot) of the returned board
 *   ep_len, ep_t         : optional run-to-termination rollout bookkeeping (ReinforceAgent.run_episode's
 *                          `while not done`, reinforce_agent.py:221-236, for a whole batch): boards with
 *                          ep_len[i] != 0 are finished and passed through untouched (reward 0); a board that
 *                          terminates or truncates in this call gets ep_len[i] = ep_t.
 */
int b2048_step_many(b2048_handle* h, const uint64_t* board_in, uint64_t* board_out,
                    uint32_t* score, uint32_t* step, uint8_t* max_exp,
                    const uint8_t* action, uint8_t* action_out, const uint8_t* flags_in,
                    const uint8_t* spawn_replay, const b2048_env_cfg* cfg /* host */,
                    int32_t* merge_sum, float* reward, double* reward64, uint8_t* flags, float* obs,
                    int32_t* ep_len, uint32_t ep_t,
                    int64_t n, uint64_t seed, uint64_t gid0, uint32_t t, void* stream);

/* n_steps consecutive b2048_step_many calls (step indices t, t + 1, ..., t + n_steps - 1) of a DEVICE-SIDE action mode
 * (random legal / random any / priority) in ONE launch, in place: every thread keeps its board, counters and legal
 * mask in registers across the steps, so the steps cost no HBM traffic, no launches and no table staging — random or
 * scripted play-outs of whole games (tools/simple_action_gen.py) are one call.  Bit-identical to the single-step calls.
 *   flags       : in/out; with flags_valid != 0 its low 4 bits are the legal masks of `board` (as left by a previous
 *                 call), else they are recomputed; on return the flags of the last step
 *   reward_last : optional, reward of the last step;  reward_sum : optional, += float32 sum of the step rewards
 *   episodes    : optional int32, += number of steps that ended an episode (meaningful with cfg->auto_reset)
 * Plain reward configuration only (base reward x scale + step reward, action mask on; score / step / max_exp all
 * given or all NULL); B2048_ERR_UNSUPPORTED otherwise. */
int b2048_step_many_n(b2048_handle* h, uint64_t* board, uint32_t* score, uint32_t* step, uint8_t* max_exp,
                      uint8_t* flags, int32_t flags_valid, const b2048_env_cfg* cfg, float* reward_last,
                      float* reward_sum, int32_t* episodes, int64_t n, int32_t n_steps, uint64_t seed,
                      uint64_t gid0, uint32_t t, void* stream);

/* Move preview without spawn (Game2048._move, game2048.py:158-165): used by the
 * differential tests and by get_action_mask-style callers. */
int b2048_move_many(b2048_handle* h, const uint64_t* board_in, uint64_t* board_out,
                    const uint8_t* action, int32_t* merge_sum, uint8_t* merge_info /* [n,4] per line */,
                    uint8_t* flags, int64_t n, void* stream);

/* The 8 dihedral variants of (board, action, legal mask): Game2048Env.get_symmetries (env.py:317-397) and
 * ReinforceAgent._augment_trajectories (reinforce_agent.py:773-808) on packed boards.  Inputs are [rows][n]
 * (any of the three may be NULL together with its output); outputs are [rows][8 n], variant v of element (r, i) at
 * r * 8n + v * n + i, variants in the reference's order (identity, three counter-clockwise quarter turns, then the
 * same four for the left-right mirror).  The upper four flag bits are copied. */
int b2048_symmetries(b2048_handle* h, const uint64_t* board, const uint8_t* flags, const uint8_t* action,
                     uint64_t* board_out, uint8_t* flags_out, uint8_t* action_out, int64_t rows, int64_t n,
                     void* stream);

/* Observation encode only (Game2048Env._preprocess_board, env.py:131-150). */
int b2048_encode_obs(const uint64_t* board, float* obs, int32_t obs_mode, float obs_log2_scale,
                     int64_t n, void* stream);

/* ---------------- policy / learner ---------------- */

enum { B2048_ACTV_SIGMOID = 0, B2048_ACTV_RELU = 1 };   /* MLP.py:130-136 */
#define B2048_MAX_LAYERS 8

/* MLP parameters as the reference stores them (MLP.py:45-94): W_l is [in_l, out_l]
 * row-major float32, b_l is [out_l].  Device pointers. */
typedef struct b2048_mlp_desc {
    int32_t n_layers;                     /* number of weight matrices (hidden + 1) */
    int32_t activation;                   /* B2048_ACTV_* */
    int32_t obs_mode;                     /* how the input vector is derived from the packed board */
    float   obs_log2_scale;
    int32_t dims[B2048_MAX_LAYERS + 1];   /* dims[0] = 16 or 272, dims[n_layers] = outputs */
    const float* W[B2048_MAX_LAYERS];
    const float* b[B2048_MAX_LAYERS];
} b2048_mlp_desc;

/* encode_observation -> forward_logits -> logits_to_probs -> sample / greedy
 * (MLP.py:22-43, :139-196; reinforce_agent.py:126-192) fused, one call for n boards.
 *   mask_flags : per-board flags byte (low 4 bits = legal mask); NULL = no mask
 *   action     : out uint8; probs/logits: optional out float32 [n, n_out]
 *   greedy     : 1 = first argmax of probs*mask (reinforce_agent.py:179-185)
 *   precision  : 0 = fp32 CUDA cores (parity path); 1 = tcgen05 tensor cores (n >= 4096): the hand-specialised bf16 kernel for the
 *                16-256-256-4 ReLU policy (raw / log2 observations), the shape-generic fp16 kernel (csrc/b2048_mlp_gen.cu) for
 *                every other ReLU policy with 1-4 hidden layers of 64 / 128 / 192 / 256 units on log2 / one-hot observations
 *                (e.g. the reference's documented one-hot [256, 128, 64] network, runner.py:27-47); B2048_ERR_UNSUPPORTED else */
int b2048_policy_step(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags,
                      const b2048_mlp_desc* mlp /* host struct, device pointers inside */,
                      uint8_t* action, float* probs, float* logits,
                      int64_t n, uint64_t seed, uint64_t gid0, uint32_t t,
                      int32_t greedy, int32_t precision, void* stream);

/* ReinforceAgent.run_episode's loop (reinforce_agent.py:221-236) for a whole batch, issued from C: n_steps times
 * { actions[t] = policy(boards[t], flags[t]); boards[t+1], flags[t+1], rewards[t] = step(boards[t], actions[t]) } for
 * t = t_begin .. t_begin + n_steps - 1.  boards / flags are time-major [T+1, B], actions / rewards [T, B].
 * ep_len != NULL: run-to-termination bookkeeping (see b2048_step_many); ep_len == NULL with cfg->auto_reset: fixed
 * horizon with reset-on-done.  t0: the env's step index before step t = 0 (Philox counter = t0 + t + 1).
 * use_mask: feed the legal masks to the policy (Game2048EnvConfig.use_action_mask).
 * precision 1 with the 16-256-256-4 ReLU policy and an action-mask-on env configuration (any reward shaping) runs the whole chunk as ONE
 * persistent kernel (tcgen05 policy + env step); anything else is a policy-kernel / step-kernel loop.
 * slot_map (device int32[n_slots], may be NULL): play only the listed boards — run-to-termination callers pass the
 * boards still alive at the start of the chunk, so finished episodes cost nothing.  Fused kernel: slices t > ep_len[b] of a
 * board that is not listed are left untouched.  Other shapes of the generic tcgen05 policy kernel (precision 1): the POLICY
 * step visits only the listed boards, the step kernel passes the finished ones through.  Anything else: B2048_ERR_INVALID.
 * n_slots_dev (device int32[1], may be NULL): the number of listed boards is read from device memory (as written by
 * b2048_compact_live) and n_slots is only an upper bound for the launch — the host can then enqueue the next chunk
 * without waiting for the count. */
int b2048_rollout_many(b2048_handle* h, uint64_t* boards, uint8_t* flags, uint8_t* actions, float* rewards,
                       uint32_t* score, uint32_t* step, uint8_t* max_exp, int32_t* ep_len,
                       const b2048_env_cfg* cfg /* host */, const b2048_mlp_desc* mlp /* host */, int64_t B,
                       int32_t t_begin, int32_t n_steps, uint64_t seed, uint64_t gid0, uint32_t t0, int32_t use_mask,
                       int32_t greedy, int32_t precision, const int32_t* slot_map, int64_t n_slots,
                       const int32_t* n_slots_dev, void* stream);

/* slot_map[0 .. *count) = the boards with ep_len[b] == 0 (episode still running), for b2048_rollout_many's slot_map;
 * count is a device int32 (zeroed by the call).  Order is unspecified (a board's results do not depend on its slot). */
int b2048_compact_live(b2048_handle* h, const int32_t* ep_len, int64_t B, int32_t* slot_map, int32_t* count,
                       void* stream);

/* ---------------- reference-seeded streams ----------------
 * The reference seeds each episode with two integers (runner.py:244-261): np.random.default_rng(env_seed) draws the
 * spawns (game2048.py:102-118) and np.random.default_rng(policy_seed) the sampled actions (rng.choice(4, p=probs),
 * reinforce_agent.py:187).  b2048_np_rng is the state of one such generator — NumPy's PCG64 with its 32-bit output
 * buffer — kept per board on the device, so that a batch plays exactly the episodes run_episode(env_seed, policy_seed)
 * plays.  Field order and meaning follow numpy's bit_generator.state: state = state_hi << 64 | state_lo,
 * inc = inc_hi << 64 | inc_lo (odd), has_uint32 / uinteger the buffered high half of the last 64-bit output. */
typedef struct b2048_np_rng {
    uint64_t state_hi, state_lo, inc_hi, inc_lo;
    uint32_t has_uint32, uinteger;
    uint64_t reserved;                    /* pads the state to 48 bytes */
} b2048_np_rng;

/* rng[i] = np.random.default_rng(seeds[i]) (PCG64 seeded through SeedSequence) for n device-side seeds in [0, 2^64). */
int b2048_np_rng_seed(const uint64_t* seeds, b2048_np_rng* rng, int64_t n, void* stream);

/* b2048_reset_many with the two spawns of Game2048.reset drawn from each board's env stream env_rng[i] (advanced in
 * place): board i is the board Game2048.reset(seed) returns when env_rng[i] = default_rng(seed).  score / step /
 * max_exp / flags as in b2048_reset_many (each may be NULL). */
int b2048_reset_many_np(b2048_handle* h, uint64_t* board, uint32_t* score, uint32_t* step, uint8_t* max_exp,
                        uint8_t* flags, b2048_np_rng* env_rng, int64_t n, void* stream);

/* b2048_rollout_many's run-to-termination loop on the reference's own random streams: the spawns of board b come from
 * env_rng[b] (as left by b2048_reset_many_np), its sampled actions from policy_rng[b] = default_rng(policy_seed)
 * (greedy = 1 draws nothing), both advanced in place; a finished board draws nothing more.  The policy is the fp32
 * CUDA-core kernel only: the tensor-core policies compute other probabilities and would therefore sample other actions.
 * ep_len is required (zero on entry for the boards still playing).  slot_map / n_slots / n_slots_dev as in
 * b2048_rollout_many (slot_map may be NULL: every board): the policy visits only the listed boards; the step kernel
 * passes the finished ones through.  Per board the result does not depend on the board's position in the batch or in
 * the list. */
int b2048_rollout_many_np(b2048_handle* h, uint64_t* boards, uint8_t* flags, uint8_t* actions, float* rewards,
                          uint32_t* score, uint32_t* step, uint8_t* max_exp, int32_t* ep_len,
                          const b2048_env_cfg* cfg /* host */, const b2048_mlp_desc* mlp /* host */, int64_t B,
                          int32_t t_begin, int32_t n_steps, b2048_np_rng* env_rng, b2048_np_rng* policy_rng,
                          int32_t use_mask, int32_t greedy, const int32_t* slot_map, int64_t n_slots,
                          const int32_t* n_slots_dev, void* stream);

/* forward_logits only (MLP.py:159-196): out[n, n_out] = logits (actor) or V(s) (critic, n_out = 1).
 *   precision : 0 = fp32 CUDA cores; 1 = single-precision tcgen05 (1e-2 class; n >= 4096: bf16 for 16-256-256-(<=4) ReLU on raw /
 *               log2 observations, fp16 on the shape-generic kernel for the other tensor-core shapes, see b2048_policy_step; else
 *               B2048_ERR_UNSUPPORTED); 3 = split-fp16 tcgen05 (every operand as fp16 hi + lo, three MMAs per product: 1e-5
 *               of the float64 result; the same shapes on log2 / one-hot observations, else B2048_ERR_UNSUPPORTED);
 *               2 = precision 3 when it applies, else fp32. */
int b2048_mlp_forward(b2048_handle* h, const uint64_t* board, const b2048_mlp_desc* mlp, float* out,
                      int64_t n, int32_t precision, void* stream);

/* forward_logits on explicit float32 inputs x[n, dims[0]] — the reference's own signature (MLP.py:159-196).
 * act_out / pre_out: HOST arrays of device pointers (either array, or any entry, may be NULL):
 * act_out[l+1] receives a_{l+1} [n, dims[l+1]] (act_out[n_layers] = logits), pre_out[l] receives z_l. */
int b2048_dense_forward(b2048_handle* h, const float* x, const b2048_mlp_desc* mlp, float* const* act_out,
                        float* const* pre_out, int64_t n, void* stream);

/* y[t] = x[t] + c * y[t+1] over t < len[b] per board, 0 beyond (compute_returns,
 * reinforce_agent.py:255-273).  x, y are [T, B] (time-major, board contiguous); len may be NULL (= T).
 * b2048_reverse_scan: one thread per board with the recurrence in float64 exactly like the reference's
 * Python loop when B >= 2048, a warp-shuffle affine suffix scan (float32) per board below that.
 * b2048_reverse_scan_f64: always the float64 per-board recurrence (bit-exact to the reference). */
int b2048_reverse_scan(const float* x, float* y, const int32_t* len, float c,
                       int32_t T, int64_t B, void* stream);
int b2048_reverse_scan_f64(const float* x, float* y, const int32_t* len, double c,
                           int32_t T, int64_t B, void* stream);

/* _compute_advantages + _compute_weighted_stats (reinforce_agent.py:276-325, :864-881) over a [T, B]
 * buffer of returns (or TD errors) v.  baseline_mode: 0 off, 1 each, 2 batch, 3 batch_norm.
 * ep_weight[B] = episode rank weights (NULL = 1).  Outputs (either may be NULL):
 *   adv[T,B]  the advantages;  coef[T,B] = adv * ep_weight[b] / (len[b] * n_traj), the per-sample weight
 *   of grad log pi in update_batch (reinforce_agent.py:533-555); both 0 for t >= len[b].
 * stats: device double[4] = {sum w, sum w v, sum w v^2, count}; computed here unless stats_precomputed != 0
 * (multi-GPU: b2048_weighted_stats on every rank, all-reduce the four doubles, then call this).
 * ep_mean_scratch: device float[B], needed for mode 1. */
int b2048_advantages(b2048_handle* h, const float* v, const int32_t* len, const float* ep_weight,
                     int32_t baseline_mode, float n_traj, int32_t T, int64_t B, float* adv, float* coef,
                     double* stats, int32_t stats_precomputed, float* ep_mean_scratch, void* stream);

/* Adds {sum w, sum w v, sum w v^2, count} over t < len[b] into stats[0..3] (_compute_weighted_stats,
 * reinforce_agent.py:864-881, as plain sums so they can be all-reduced across ranks). */
int b2048_weighted_stats(b2048_handle* h, const float* v, const int32_t* len, const float* ep_weight,
                         int32_t T, int64_t B, double* stats, void* stream);

/* TD(0) errors of the critic block (reinforce_agent.py:439-447): td = r + gamma V(s') [t+1 < len] - V(s);
 * gcoef = dLoss/dV * ep_weight/(len n_traj) with dLoss/dV = V - target (mse) or its Huber clip
 * (_get_grad_logits_critic, reinforce_agent.py:884-910).  All buffers [T, B]. */
int b2048_td_errors(b2048_handle* h, const float* reward, const float* value, const int32_t* len,
                    const float* ep_weight, float gamma, int32_t huber, float huber_delta, float n_traj,
                    int32_t T, int64_t B, float* td, float* gcoef, void* stream);

/* ---------------- fixed-horizon windows ----------------
 * A window is a b2048_rollout_many fixed-horizon rollout with reset-on-done: T steps of B lanes, a lane holds several
 * episodes.  e[t,b] = (flags[t+1,b] & (B2048_F_DONE | B2048_F_TRUNC)) != 0 ends an episode at step t (boards[t+1] is
 * the reset board); a truncated episode is not bootstrapped, like update_batch's last step. */

/* Per-lane targets of a window (one thread per lane, float64 recurrence).  rewards [T,B], flags [T+1,B].
 *   value == NULL (REINFORCE): v = G_t = r_t + gamma (1 - e_t) G_{t+1}; valid_len[b] = 1 + the lane's last boundary (0 if
 *                none): later slots belong to an episode that does not end in the window, and v is 0 there.
 *   value [T+1,B] (actor-critic, V(boards[t]) for every slice): td = delta_t = r_t + gamma (1 - e_t) V_{t+1} - V_t (V_T
 *                bootstraps the cut-off tail); v = A_t = delta_t + gamma lambda (1 - e_t) A_{t+1}; gcoef = dLoss/dV of
 *                delta (mse, or its Huber clip with huber != 0, _get_grad_logits_critic) / (T n_traj); valid_len = T.
 * td / gcoef are required with a value and unused without. */
int b2048_segment_targets(b2048_handle* h, const float* reward, const uint8_t* flags, const float* value, double gamma,
                          double lambda, int32_t huber, float huber_delta, float n_traj, int32_t T, int64_t B, float* v,
                          float* td, float* gcoef, int32_t* valid_len, void* stream);

/* b2048_advantages for a window: the samples of lane b are t < valid_len[b] and coef = adv / (T n_traj) (an episode's
 * length is not known inside a window).  baseline_mode 0 off, 2 batch, 3 batch_norm; stats / stats_precomputed as in
 * b2048_advantages (b2048_weighted_stats with len = valid_len gives the sums). */
int b2048_advantages_window(b2048_handle* h, const float* v, const int32_t* valid_len, int32_t baseline_mode, float n_traj,
                            int32_t T, int64_t B, float* adv, float* coef, double* stats, int32_t stats_precomputed,
                            void* stream);

/* Episodes completed inside a window, for logging.  ep_return[B] (device double, in/out) carries the undiscounted return
 * of each lane's running episode from window to window (zero it with the reset).  Each episode that ends in the window
 * is ADDED into stats (device double[21]) = {count, sum of returns, max (init -inf), min (init +inf), then 17 counts by
 * the exponent of its max tile}: max(4, the largest tile after its last move, boards[t] with actions[t]), 16 for a
 * 32768+32768 merge.  boards [T+1,B] (slices 0..T-1 read), actions [T,B]. */
int b2048_horizon_episodes(b2048_handle* h, const float* reward, const uint8_t* flags, const uint64_t* board,
                           const uint8_t* action, int32_t T, int64_t B, double* ep_return, double* stats, void* stream);

/* Bootstrapping at truncation.  A TRUNC flag ends an episode only because the step budget ran out, so the episode's last
 * target is r + gamma V(s'), with s' the board the episode was cut on.
 *
 * b2048_replay_pre_reset: s' of a fixed-horizon window played with auto-reset (where boards[t + 1] already holds the reset
 * board).  For each listed slot s = t * B + b of the [T, B] window, out[k] = the board after actions[s] on boards[s] and the
 * Philox spawn of (seed, gid0 + b, t0 + t + 1) -- the counter b2048_rollout_many used for that step -- with no spawn when
 * the move changed nothing.  It is the step body with auto-reset off, so it equals b2048_step_many on the same inputs.
 * boards [T+1, B], actions [T, B], slots [K] (device, int64, each >= 0 and < T * B), out [K] (device).  The slot list is
 * checked on the host: the call waits for `stream`.
 *
 * b2048_fold_bootstrap: reward_out[i] = reward[i] for i in [0, n), except reward_out[slots[k]] = reward[slots[k]] +
 * gamma * value[k] with the multiply and the add rounded separately.  Fed to b2048_segment_targets or b2048_td_errors,
 * whose target at an episode's last step is r + gamma * 0, this gives the bootstrapped target, TD error, advantage and
 * critic coefficient bit for bit.  slots [K] distinct and in [0, n) (checked on the host: the call waits for `stream`);
 * reward_out may be reward. */
int b2048_replay_pre_reset(b2048_handle* h, const uint64_t* boards, const uint8_t* actions, const int64_t* slots, int64_t K,
                           int64_t B, uint64_t seed, uint64_t gid0, uint32_t t0, uint64_t* out, void* stream);
int b2048_fold_bootstrap(b2048_handle* h, const float* reward, const int64_t* slots, const float* value, int64_t K, int64_t n,
                         float gamma, float* reward_out, void* stream);

/* Gradient accumulation of update_batch's actor / critic blocks (reinforce_agent.py:403-555, _backpropagation
 * :639-678) over n samples (flattened [T,B] rollout; samples with coef == 0 contribute nothing).
 * grads is a flat float32 vector laid out W_0, b_0, W_1, b_1, ... and is ACCUMULATED into (zero it first).
 *   head_mode 0: += d/dtheta sum_s coef[s] log pi(action[s] | board[s])   (mask_flags: legal masks, may be NULL)
 *   head_mode 1: += d/dtheta sum_s coef[s] V(board[s])
 * workspace: device floats, at least b2048_backward_workspace_floats(mlp, chunk); samples are processed
 * `chunk` at a time.
 *   precision : 0 = fp32 CUDA cores;
 *               3 = float32-grade tensor-core path (n >= 4096; 16-256-256-(<=4) ReLU on log2 observations: the persistent
 *                   update pipeline; every other ReLU network with 1-4 hidden layers of 64 / 128 / 192 / 256 units on log2 /
 *                   one-hot observations: gen_mlp_kernel + gen_dw_kernel; anything else returns B2048_ERR_UNSUPPORTED):
 *                   forward with split-fp16 operands (hi + lo, three tcgen05.mma per product), backward deltas and dW GEMMs
 *                   in fp16 with a power-of-two loss scale, fp32 accumulation.
 *                   Within 1e-2 of the float32 gradient also on heavily cancelling (zero-mean advantage) batches;
 *               2 = precision 3 when it applies, else fp32 (what the host layer's "auto" passes);
 *               1 = single-bf16 tensor cores (raw / log2 observations), an explicit opt-in: its forward pass flips ReLU
 *                   units whose pre-activation is within bf16 rounding of zero, a 3-30 % error on cancelling gradients. */
int64_t b2048_backward_workspace_floats(const b2048_mlp_desc* mlp, int64_t chunk);
int b2048_mlp_backward(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags,
                       const uint8_t* action, const float* coef, const b2048_mlp_desc* mlp, float* grads,
                       int64_t n, int32_t head_mode, float* workspace, int64_t workspace_floats,
                       int64_t chunk, int32_t precision, void* stream);
/* Test / debug access to the tensor-core path's workspace: byte offsets (from the workspace pointer rounded up to
 * 1024 B) of the bf16 images H1, H2, DL2, DL1 ([64-sample tile][4 feature slabs][64 rows][128 B, 128-byte
 * swizzle]) and A1^T, d3^T ([tile][16 rows][128 B]), then the total. */
int b2048_backward_tc_layout(int64_t chunk, int64_t* out7);

/* clip_grads_global_norm (reinforce_agent.py:835-861) + SGD (:565-575) or Adam (:719-770) on a flat parameter
 * vector.  optimizer 0 sgd / 1 adam; sign +1 ascent (actor), -1 descent (critic); adam_t = step count after
 * increment.  grads is clipped in place; sumsq_out (device double[1]) receives the squared norm before clipping. */
int b2048_apply_update(b2048_handle* h, float* theta, float* grads, float* adam_m, float* adam_v, int64_t n,
                       int32_t optimizer, float lr, float sign, float max_grad_norm, float beta1, float beta2,
                       int32_t adam_t, double* sumsq_out, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2048_H_ */
