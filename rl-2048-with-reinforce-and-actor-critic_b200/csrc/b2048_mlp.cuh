// b2048_mlp.cuh — fp32 CUDA-core MLP tile shared by the policy-step, value-forward and backward
// kernels (the parity path; the bf16 tcgen05 path lives in b2048_policy_tc.cu).
//
// A CTA of 256 threads owns a tile of kTileM = 64 boards.  Activations of every layer stay in shared
// memory as [board][dim + 4] float32 (the +4 pad keeps 128-bit rows aligned and de-conflicts the
// head's per-board reads).  Warp w owns boards 8w..8w+7, lane owns columns lane + 32 j: weight reads
// are 128-byte coalesced through L1 (the whole net is 285 KB and L2/L1 resident), activation reads
// are warp-broadcast LDS.128, every thread keeps an 8 x 8 register tile.
//
// Reference arithmetic restated: forward_logits z = a @ W + b, Sigmoid / ReLU hidden, linear head
// (src/MLP.py:130-136, :159-196); encode_observation flatten order (r*4+c)[*17+e] (src/MLP.py:22-43,
// src/env.py:131-150); W is [in, out] row-major exactly as the reference stores it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/b2048.h"

namespace b2 {

constexpr int kTileM = 64;
constexpr int kMlpThreads = 256;
constexpr int kPad = 4;

struct MlpDev {
    int n_layers, activation, obs_mode;
    float obs_scale;
    int dims[B2048_MAX_LAYERS + 1];
    const float* W[B2048_MAX_LAYERS];
    const float* b[B2048_MAX_LAYERS];
};

// float offset of layer-l input activations inside the shared activation arena
__host__ __device__ inline int act_offset(const int* dims, int l) {
    int off = 0;
    for (int i = 0; i < l; ++i) off += kTileM * ((i == 0 ? 16 : dims[i]) + kPad);
    return off;
}
__host__ __device__ inline int act_stride(const int* dims, int l) { return (l == 0 ? 16 : dims[l]) + kPad; }

__device__ __forceinline__ float activate(float z, int mode) {
    return mode == B2048_ACTV_RELU ? fmaxf(z, 0.0f) : 1.0f / (1.0f + expf(-z));
}
// derivative expressed through the activation value a = act(z) (reinforce_agent.py:624-636)
__device__ __forceinline__ float activate_grad(float a, int mode) {
    return mode == B2048_ACTV_RELU ? (a > 0.0f ? 1.0f : 0.0f) : a * (1.0f - a);
}

// Layer-0 input rows: raw / log2 -> 16 floats; onehot -> 16 exponents stored as int bits.
// slots != NULL: row s of the tile is board slots[s] (a live-board list), else board s.
__device__ __forceinline__ void encode_input(float* x0 /*[kTileM][16+pad]*/, const uint64_t* __restrict__ board,
                                             int64_t s0, int64_t n, int obs_mode, float scale,
                                             const int32_t* __restrict__ slots = nullptr) {
    for (int idx = threadIdx.x; idx < kTileM * 16; idx += kMlpThreads) {
        int b = idx >> 4, cell = idx & 15;
        int64_t s = s0 + b;
        uint32_t e = 0;
        if (s < n) e = (uint32_t)((board[slots ? (int64_t)slots[s] : s] >> (4 * cell)) & 0xFull);
        float v;
        if (obs_mode == B2048_OBS_ONEHOT) v = __int_as_float((int)e);
        else if (obs_mode == B2048_OBS_RAW) v = e ? (float)(1u << e) : 0.0f;
        else v = (float)e * scale;
        x0[b * (16 + kPad) + cell] = v;
    }
}

// out[b][c] = act( bias[c] + sum_k A[b][k] * W[k][c] )    A: smem [kTileM][K+pad], W: global [K][N]
// kEpi: 0 = store act(z) to Out (and optionally to gout[s][N]);
//       1 = backward: multiply by act'(Out_old) in place (Out holds a_l), store to Out and gout.
template <int kEpi>
__device__ __forceinline__ void tile_layer(const float* __restrict__ A, int K, int a_stride, const float* __restrict__ W,
                                           const float* __restrict__ bias, int N, float* __restrict__ Out, int o_stride,
                                           int act_mode, bool apply_act, float* __restrict__ gout, int64_t s0, int64_t n,
                                           float* __restrict__ gpre = nullptr) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const float* Aw = A + (warp * 8) * a_stride;
    for (int c0 = 0; c0 < N; c0 += 256) {
        float acc[8][8];
#pragma unroll
        for (int b = 0; b < 8; ++b)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[b][j] = 0.0f;
        for (int k0 = 0; k0 < K; k0 += 4) {
            float4 a[8];
#pragma unroll
            for (int b = 0; b < 8; ++b) a[b] = *reinterpret_cast<const float4*>(Aw + b * a_stride + k0);
#pragma unroll
            for (int kk = 0; kk < 4; ++kk) {
                float w[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    int c = c0 + j * 32 + lane;
                    w[j] = c < N ? __ldg(W + (size_t)(k0 + kk) * N + c) : 0.0f;
                }
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    float av = kk == 0 ? a[b].x : kk == 1 ? a[b].y : kk == 2 ? a[b].z : a[b].w;
#pragma unroll
                    for (int j = 0; j < 8; ++j) acc[b][j] = fmaf(av, w[j], acc[b][j]);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int c = c0 + j * 32 + lane;
            if (c < N) {
                float bv = bias ? __ldg(bias + c) : 0.0f;
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    int row = warp * 8 + b;
                    float z = acc[b][j] + bv;
                    float v;
                    if (kEpi == 0) v = apply_act ? activate(z, act_mode) : z;
                    else v = z * activate_grad(Out[row * o_stride + c], act_mode);
                    Out[row * o_stride + c] = v;
                    if (gout != nullptr && s0 + row < n) gout[(s0 + row) * N + c] = v;
                    if (gpre != nullptr && s0 + row < n) gpre[(s0 + row) * N + c] = z;
                }
            }
        }
    }
}

// Layer 0 for one-hot input: z[c] = bias[c] + sum_cell W[cell*17 + e_cell][c]  (a 16-row gather-sum of
// W0 instead of a 272-long dot product: the one-hot first layer is exactly that).
__device__ __forceinline__ void tile_layer0_onehot(const float* __restrict__ X0, const float* __restrict__ W,
                                                   const float* __restrict__ bias, int N, float* __restrict__ Out,
                                                   int o_stride, int act_mode, bool apply_act, float* __restrict__ gout,
                                                   int64_t s0, int64_t n) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int xs = 16 + kPad;
    for (int c0 = 0; c0 < N; c0 += 256) {
        float acc[8][8];
#pragma unroll
        for (int b = 0; b < 8; ++b)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[b][j] = 0.0f;
        for (int cell = 0; cell < 16; ++cell) {
#pragma unroll
            for (int b = 0; b < 8; ++b) {
                int e = __float_as_int(X0[(warp * 8 + b) * xs + cell]);
                const float* wr = W + (size_t)(cell * 17 + e) * N;
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    int c = c0 + j * 32 + lane;
                    if (c < N) acc[b][j] += __ldg(wr + c);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            int c = c0 + j * 32 + lane;
            if (c < N) {
                float bv = __ldg(bias + c);
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    int row = warp * 8 + b;
                    float z = acc[b][j] + bv;
                    float v = apply_act ? activate(z, act_mode) : z;
                    Out[row * o_stride + c] = v;
                    if (gout != nullptr && s0 + row < n) gout[(s0 + row) * N + c] = v;
                }
            }
        }
    }
}

// Forward through all hidden layers of the tile; activations of layer l input live at
// arena + act_offset(l).  If gact != nullptr, hidden activations a_l (l >= 1) are also written to
// gact[l][s][dim_l] for the weight-gradient GEMMs.  Ends with __syncthreads().
__device__ __forceinline__ void tile_forward_hidden(float* arena, const MlpDev& m, const uint64_t* __restrict__ board,
                                                    int64_t s0, int64_t n, float* const* gact,
                                                    const int32_t* __restrict__ slots = nullptr) {
    encode_input(arena, board, s0, n, m.obs_mode, m.obs_scale, slots);
    __syncthreads();
    const int L = m.n_layers;
    for (int l = 0; l + 1 < L; ++l) {
        float* in = arena + act_offset(m.dims, l);
        float* out = arena + act_offset(m.dims, l + 1);
        float* g = gact ? gact[l + 1] : nullptr;
        if (l == 0 && m.obs_mode == B2048_OBS_ONEHOT)
            tile_layer0_onehot(in, m.W[0], m.b[0], m.dims[1], out, act_stride(m.dims, 1), m.activation, true, g, s0, n);
        else
            tile_layer<0>(in, l == 0 ? 16 : m.dims[l], act_stride(m.dims, l), m.W[l], m.b[l], m.dims[l + 1], out,
                          act_stride(m.dims, l + 1), m.activation, true, g, s0, n);
        __syncthreads();
    }
}

// Linear head (n_out <= 4): thread t -> board t/4, output t%4 (or a quarter of K when n_out == 1).
// Returns this thread's output (valid for j < n_out; for n_out == 1 every lane of the quad holds it).
__device__ __forceinline__ float tile_head(const float* arena, const MlpDev& m) {
    const int L = m.n_layers;
    const int b = threadIdx.x >> 2, j = threadIdx.x & 3;
    const int n_out = m.dims[L];
    const float* W = m.W[L - 1];
    float acc = 0.0f;
    if (L == 1 && m.obs_mode == B2048_OBS_ONEHOT) {
        const float* x = arena + b * (16 + kPad);
        if (n_out == 1) {
            for (int cell = j; cell < 16; cell += 4) acc += __ldg(W + (cell * 17 + __float_as_int(x[cell])));
            acc += __shfl_xor_sync(0xFFFFFFFFu, acc, 1);
            acc += __shfl_xor_sync(0xFFFFFFFFu, acc, 2);
        } else if (j < n_out) {
            for (int cell = 0; cell < 16; ++cell) acc += __ldg(W + (size_t)(cell * 17 + __float_as_int(x[cell])) * n_out + j);
        }
    } else {
        const int K = (L == 1) ? 16 : m.dims[L - 1];
        const float* a = arena + act_offset(m.dims, L - 1) + b * act_stride(m.dims, L - 1);
        if (n_out == 1) {
            for (int k = j; k < K; k += 4) acc = fmaf(a[k], __ldg(W + k), acc);
            acc += __shfl_xor_sync(0xFFFFFFFFu, acc, 1);
            acc += __shfl_xor_sync(0xFFFFFFFFu, acc, 2);
        } else if (j < n_out) {
            for (int k = 0; k < K; ++k) acc = fmaf(a[k], __ldg(W + (size_t)k * n_out + j), acc);
        }
    }
    int jb = n_out == 1 ? 0 : j;
    if (jb < n_out) acc += __ldg(m.b[L - 1] + jb);
    return acc;
}

// logits_to_probs (src/MLP.py:139-156) across the 4 lanes of a quad: masked fill -1e9, max-subtracted softmax.
__device__ __forceinline__ float quad_softmax(float logit, bool legal, bool use_mask) {
    float l = (use_mask && !legal) ? -1e9f : logit;
    float mx = fmaxf(l, __shfl_xor_sync(0xFFFFFFFFu, l, 1));
    mx = fmaxf(mx, __shfl_xor_sync(0xFFFFFFFFu, mx, 2));
    float e = expf(l - mx);
    float s = e + __shfl_xor_sync(0xFFFFFFFFu, e, 1);
    s = s + __shfl_xor_sync(0xFFFFFFFFu, s, 2);
    return e / s;
}

inline size_t mlp_arena_bytes(const int* dims, int n_layers) {
    return (size_t)act_offset(dims, n_layers) * sizeof(float) + (size_t)kTileM * 4 * sizeof(float);
}

}  // namespace b2
