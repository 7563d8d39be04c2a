// b2048_mlp_gen.cu — the tensor-core MLP kernels for EVERY layer shape the reference's generic MLP is configured with
// (src/MLP.py:45-94, :159-196: any number of hidden layers, one-hot 272-wide or 16-wide input), in particular its
// documented one-hot [256, 128, 64] configuration (runner.py:27-47).  The kernels of b2048_policy_tc.cu / b2048_learn_hp.cu
// are hand-specialised for the runner-default 16-256-256-4 network; these are shape-generic:
//
//  gen_mlp_kernel    one persistent CTA per SM walks 128-sample tiles; per tile it runs a short PROGRAM of GEMMs on
//                    tcgen05: the forward layers and — for an update — the head delta (masked softmax / value head, I/O
//                    warps) and the backward delta GEMMs, all in one launch.  Activations never leave the SM between
//                    layers: every GEMM's epilogue (16 warps: TMEM -> bias / ReLU / mask -> fp16) writes the next GEMM's A
//                    operand into one 128 KB shared-memory buffer of 128-byte-swizzled K-major slabs.  The weights do not
//                    fit next to it (the one-hot network's split image is 444 KB), so they STREAM: a loader lane pulls
//                    64-wide K-slab units [N rows x 128 B] from the L2-resident image through a 3-slot ring of bulk copies.
//                    Forward precision: every product is three MMAs on fp16 hi + lo operands (float32 grade; the one-hot /
//                    log2 inputs are exact in fp16, so layer 0 needs two), or one MMA (rollout policy steps).  Backward:
//                    fp16 deltas with a power-of-two loss scale, as in b2048_learn_hp.cu.  For the dW GEMMs the hi halves of
//                    the activations and the deltas leave as slab images (bulk shared -> global copies by the MMA lane).
//  gen_mlp_ent_kernel  gen_mlp_kernel in update mode with the entropy bonus in the policy head's delta (b2048_entropy.cuh)
//  gen_dw_kernel     dW_l = A_{l-1}^T DL_l (_backpropagation, src/reinforce_agent.py:639-678) for one layer: the slab
//                    images are read back MN-major; split over 128-feature M tiles and sample ranges; the one-hot / log2
//                    input of layer 0 is regenerated from the packed boards in shared memory instead of being stored.
#include <cuda_fp16.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstring>

#include "b2048_device.cuh"
#include "b2048_entropy.cuh"
#include "b2048_internal.h"
#include "b2048_tc.cuh"

namespace b2 {

constexpr int GN_MAXL = 5;                     // weight matrices: up to 4 hidden layers + the head
constexpr int GN_MAXU = 64;                    // streamed weight units per tile
constexpr int GN_MAXG = 2 * GN_MAXL - 1;       // GEMMs per tile (forward + backward)
constexpr int GN_SLAB = 16384;                 // [128 rows x 128 B], SWIZZLE_128B: 64 features of 128 samples
constexpr int GN_SLOT = 32768;                 // weight ring slot: one unit of up to 256 rows x 128 B
constexpr int GN_NSLOT = 3;
constexpr int GS_A = 0;                        // A buffer: hi slabs 0..3, lo slabs 4..7 (a 272-wide input uses slabs 0..4)
constexpr int GS_W = 8 * GN_SLAB;
constexpr int GS_BAR = GS_W + GN_NSLOT * GN_SLOT;
constexpr int GS_ONES = GS_BAR + 256;          // constant A operand of the bias MMAs: every row = e0 + e1 (fp16), 256 B
constexpr int GS_TOTAL = GS_ONES + 256;
constexpr int GN_THREADS = 22 * 32;            // 16 epilogue warps, MMA warp, weight loader, 4 I/O warps
constexpr int GN_MASK_WORDS = 4 * 4 * 4 * 128; // per CTA: [hidden layer][slab][column group][row] 16-bit ReLU masks
static_assert(GS_TOTAL <= 232448, "gen_mlp_kernel exceeds the shared memory of an sm_100 CTA");

struct GUnit {            // one streamed weight unit = the B operand of up to 8 MMAs
    uint32_t off;         // byte offset inside the weight image
    uint16_t rows;        // B rows (the MMA's N); bytes = rows * 128
    uint8_t layer, slab;  // weight matrix, 64-wide K slab
    uint8_t ksteps;       // valid K = 16 steps of the slab (1..4)
    uint8_t kind;         // 0: forward hi, 1: forward lo, 2: backward (fp16 W read as [in][out]), 3: bias [rows x 16] (k = 0: hi, 1: lo)
    uint16_t bytes16;     // unit size / 16
    uint16_t slot_off16;  // offset of the unit inside its ring slot / 16
    uint16_t pad;
};
struct GFill {            // consecutive units of one GEMM that travel in ONE ring slot (<= 32 KB): one bulk load, one slot release.
    uint32_t off;         // A tcgen05.commit drains the MMA pipeline (~400 cycles measured), so slots are released per fill, not per unit
    uint16_t bytes16;
    uint8_t u0, nu;
};
struct GGemm {
    uint8_t f0, nf;       // its fills (ring slots)
    uint8_t u0, nu;       // its units
    uint8_t layer, bwd;   // forward: z_layer = a_{layer-1} W_layer;  backward: delta_{layer-1} = delta_layer W_layer^T
    uint16_t N;           // accumulator columns
    uint8_t a_lo;         // the A operand has a lo half (split forward, layer > 0)
    uint8_t head;         // forward head GEMM: read by the I/O warps
    uint8_t from_io;      // its A operand is written by the I/O warps (the tile's input; the head deltas)
    uint8_t pad;
};
// Per-unit issue record of the MMA warp (tile-invariant; lane l keeps records l and l + 32 in registers, a shuffle broadcasts one):
// [0..15] offset in the ring slot / 16, [16..18] K steps, [19..20] kind, [21] first unit of its fill, [22] last unit of its fill,
// [23] first unit of a K slab written by the epilogue warps (wait for the slab), [24..26] K slab, [27] the slab leaves as an image
constexpr uint32_t GR_FIRST = 1u << 21, GR_LAST = 1u << 22, GR_SLABWAIT = 1u << 23, GR_STORE = 1u << 27, GR_LOPART = 1u << 28;
struct GenProg {
    GUnit unit[GN_MAXU];
    GFill fill[GN_MAXU];
    GGemm gemm[GN_MAXG];
    uint32_t rec[GN_MAXU];
    int n_units, n_fills, n_gemm, L, fb, split;
    int kin, in_slabs, obs_mode, n_out;
    int act;              // B2048_ACTV_RELU / B2048_ACTV_SIGMOID (MLP.py:130-136)
    float obs_scale;
    int width[GN_MAXL];   // accumulator width of layer l (hidden: its size; head: 16)
    uint32_t img_bytes;
};


// ---- the program builder: constexpr, so that the host builds the table-driven program of ANY supported network with it and the
//      kernel can be instantiated with the program of one network as compile-time constants (straight-line MMA issue, see SpecProg)
struct NetDims { int L, kin, obs_mode, n_out, act; int hid[GN_MAXL]; };

// packs the units [u0, u1) of GEMM G (contiguous in the image) into ring-slot fills of at most GN_SLOT bytes
__host__ __device__ constexpr void pack_fills(GenProg& p, int G, int u0, int u1) {
    GGemm& g = p.gemm[G];
    g.f0 = (uint8_t)p.n_fills; g.u0 = (uint8_t)u0; g.nu = (uint8_t)(u1 - u0);
    int u = u0;
    while (u < u1) {
        GFill& f = p.fill[p.n_fills++];
        f.off = p.unit[u].off; f.u0 = (uint8_t)u;
        uint32_t bytes = 0;
        while (u < u1) {
            const uint32_t start = p.unit[u].off - f.off, ub = (uint32_t)p.unit[u].bytes16 * 16u;
            if (start + ub > (uint32_t)GN_SLOT) break;
            p.unit[u].slot_off16 = (uint16_t)(start / 16u);
            bytes = start + ub;
            ++u;
        }
        f.nu = (uint8_t)(u - f.u0); f.bytes16 = (uint16_t)(bytes / 16u);
    }
    g.nf = (uint8_t)(p.n_fills - g.f0);
    g.from_io = (G == 0 || (g.bwd && G == p.L)) ? 1 : 0;
    for (int f = g.f0; f < g.f0 + g.nf; ++f) {
        const GFill& fl = p.fill[f];
        for (int k = fl.u0; k < fl.u0 + fl.nu; ++k) {
            const GUnit& un = p.unit[k];
            uint32_t r = (uint32_t)un.slot_off16 | ((uint32_t)un.ksteps << 16) | ((uint32_t)un.kind << 19) | ((uint32_t)un.slab << 24);
            if (k == fl.u0) r |= GR_FIRST;
            if (k == fl.u0 + fl.nu - 1) r |= GR_LAST;
            const bool slab_first = un.kind == 0 || un.kind == 2;
            if (slab_first && !g.from_io) r |= GR_SLABWAIT;
            if (slab_first && p.fb && G > 0) r |= GR_STORE;
            if (un.kind == 0 && g.a_lo) r |= GR_LOPART;
            p.rec[k] = r;
        }
    }
}

__host__ __device__ constexpr GenProg make_prog(const NetDims& d, bool split, bool fb) {
    GenProg p{};
    const int L = d.L;
    p.L = L; p.fb = fb ? 1 : 0; p.split = split ? 1 : 0;
    p.kin = d.kin; p.in_slabs = (p.kin + 63) / 64; p.obs_mode = d.obs_mode; p.n_out = d.n_out;
    p.obs_scale = 1.0f;
    p.act = d.act;
    for (int l = 0; l < L; ++l) p.width[l] = l == L - 1 ? 16 : d.hid[l];
    uint32_t off = 0;
    int nu = 0, ng = 0;
    for (int l = 0; l < L; ++l) {            // forward
        const int K = l == 0 ? d.kin : d.hid[l - 1], slabs = (K + 63) / 64;
        const int G = ng++;
        GGemm& g = p.gemm[G];
        const int g_u0 = nu;
        g.layer = (uint8_t)l; g.bwd = 0; g.N = (uint16_t)p.width[l]; g.a_lo = (split && l > 0) ? 1 : 0;
        g.head = l == L - 1 ? 1 : 0;
        for (int s = 0; s < slabs; ++s) {
            const int ks = (K - 64 * s) >= 64 ? 4 : (K - 64 * s + 15) / 16;
            for (int part = 0; part < (split ? 2 : 1); ++part) {
                GUnit& u = p.unit[nu++];
                u.off = off; u.rows = (uint16_t)p.width[l]; u.layer = (uint8_t)l; u.slab = (uint8_t)s; u.ksteps = (uint8_t)ks;
                u.kind = (uint8_t)part;
                u.bytes16 = (uint16_t)(ks == 1 ? u.rows * 2 : u.rows * 8);     // a single-K-step unit is stored compactly (K = 16 only)
                off += (uint32_t)u.bytes16 * 16u;
            }
        }
        if (l < L - 1) {                     // hidden layers: the bias comes in through one more MMA (head: added by the I/O warps)
            GUnit& u = p.unit[nu++];
            u.off = off; u.rows = (uint16_t)p.width[l]; u.layer = (uint8_t)l; u.slab = 0; u.ksteps = 1; u.kind = 3;
            u.bytes16 = (uint16_t)(u.rows * 2);
            off += (uint32_t)u.rows * 32u;
        }
        pack_fills(p, G, g_u0, nu);
        off = (off + 1023u) & ~1023u;
    }
    if (fb) {
        for (int l = L - 1; l >= 1; --l) {   // delta_{l-1} = delta_l W_l^T: K = width of layer l, rows = width of layer l - 1
            const int Kp = p.width[l], slabs = (Kp + 63) / 64;
            const int G = ng++;
            GGemm& g = p.gemm[G];
            const int g_u0 = nu;
            g.layer = (uint8_t)l; g.bwd = 1; g.N = (uint16_t)p.width[l - 1]; g.a_lo = 0; g.head = 0;
            for (int s = 0; s < slabs; ++s) {
                GUnit& u = p.unit[nu++];
                u.off = off; u.rows = (uint16_t)p.width[l - 1]; u.layer = (uint8_t)l; u.slab = (uint8_t)s;
                u.ksteps = (uint8_t)((Kp - 64 * s) >= 64 ? 4 : (Kp - 64 * s + 15) / 16);
                u.kind = 2;
                u.bytes16 = (uint16_t)(u.ksteps == 1 ? u.rows * 2 : u.rows * 8);
                off += (uint32_t)u.bytes16 * 16u;
            }
            pack_fills(p, G, g_u0, nu);
        }
    }
    p.n_units = nu; p.n_gemm = ng; p.img_bytes = off;
    return p;
}

// Programs known at compile time: kSpec 1 = the reference's documented one-hot 272-256-128-64 network (runner.py:27-47).
template <int kSpec, bool kSplit, bool kFb> struct SpecProg;
template <bool kSplit, bool kFb> struct SpecProg<1, kSplit, kFb> {
    static constexpr NetDims D{4, 272, B2048_OBS_ONEHOT, 4, B2048_ACTV_RELU, {256, 128, 64, 0, 0}};
    static constexpr GenProg P = make_prog(D, kSplit, kFb);
};

struct GenArgs {
    GenProg p;
    const float* bias[GN_MAXL];
    const uint8_t* img;
    const uint64_t* board;
    int64_t n;
    // ---- forward-only outputs (each nullable)
    float* out;                 // [n][n_out] head outputs
    uint8_t* action;
    float* probs;
    float* logits;
    const uint8_t* mask_flags;  // legal masks (sampling and the policy head's softmax)
    const int32_t* slot_map;    // policy steps of a run-to-termination rollout: sample s is board slot_map[s] (NULL: s)
    const int32_t* n_dev;       // with slot_map: the number of listed boards, read on the device (NULL: n)
    PhiloxKeys keys;
    uint64_t gid0;
    uint32_t t;
    int greedy;
    // ---- update mode (p.fb)
    const uint8_t* act_in;
    const float* coef;
    const float* scale;         // device float[2]: loss scale S and 1 / S
    int head_mode;
    uint8_t* himg[GN_MAXL];     // hi activation images a_{l+1} of the hidden layers, [tile][slab][128 x 128 B]
    uint8_t* dlimg[GN_MAXL];    // delta images of every layer (head: one slab)
    float* gb_head;
    uint16_t* mask_scratch;     // [grid][GN_MASK_WORDS]  (ReLU)
    uint4* dsig_scratch;        // [grid][GN_MASK_WORDS][2]: s (1 - s) of every hidden unit as fp16 (Sigmoid, update mode)
    long long* dbg;             // optional phase clocks of CTA 0 (B2048_DBG_TC_CLOCKS), 64 slots per tile for the first 4 tiles
};

__device__ __forceinline__ void g_bulk_store(uint8_t* dst, uint32_t src, uint32_t bytes) {
    for (uint32_t off = 0; off < bytes; off += 16384u) bulk_store(dst + off, src + off, 16384u);
}

// Row `row` of the network input as fp16 K-major slab rows: slabs slab0 .. slab0 + nslabs - 1 of the input go to dst,
// dst + GN_SLAB, ...  one-hot: feature cell * 17 + exponent (env.py:131-150) — the caller has zero-filled the slabs (linearly:
// a per-row fill would be an 8-way bank conflict); log2: exponent * scale in the first 16 features (nothing else is read).
__device__ __forceinline__ void zero_slabs_128(uint8_t* dst, int nslabs, int t128) {
    for (int i = t128; i < nslabs * (GN_SLAB / 16); i += 128) *reinterpret_cast<uint4*>(dst + i * 16) = make_uint4(0u, 0u, 0u, 0u);
}
__device__ __forceinline__ void encode_input_row(uint64_t bd, int row, uint8_t* dst, int slab0, int nslabs, int obs_mode,
                                                 float scale) {
    const int sw = row & 7;
    if (obs_mode == B2048_OBS_ONEHOT) {
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const int f = c * 17 + (int)((bd >> (4 * c)) & 0xFull);
            const int s = (f >> 6) - slab0, k = f & 63;
            if (s >= 0 && s < nslabs)
                *reinterpret_cast<uint16_t*>(dst + s * GN_SLAB + row * 128 + (((k >> 3) ^ sw) << 4) + (k & 7) * 2) = 0x3C00u;   // 1.0
        }
    } else if (slab0 == 0) {
#pragma unroll
        for (int c = 0; c < 16; ++c) {
            const float v = (float)((uint32_t)(bd >> (4 * c)) & 0xFu) * scale;
            *reinterpret_cast<__half*>(dst + row * 128 + (((c >> 3) ^ sw) << 4) + (c & 7) * 2) = __float2half_rn(v);
        }
    }
}

// ------------------------------------------------------------------------------------------------ weight image
struct GenPrepArgs {
    GenProg p;
    const float* W[GN_MAXL];
    const float* b[GN_MAXL];
    int dims[GN_MAXL + 1];
    uint8_t* img;
};
__global__ void __launch_bounds__(256) gen_prepare_kernel(const __grid_constant__ GenPrepArgs a) {
    const int tid = blockIdx.x * blockDim.x + threadIdx.x, nth = gridDim.x * blockDim.x;
    for (int u = 0; u < a.p.n_units; ++u) {
        const GUnit un = a.p.unit[u];
        const int K = a.dims[un.layer], N = a.dims[un.layer + 1];
        const float* W = a.W[un.layer];
        if (un.kind == 3) {                 // [rows / 8][2 k-chunks][8 rows][16 B], no swizzle: k = 0 -> hi(b[n]), k = 1 -> lo(b[n]), rest 0
            for (int idx = tid; idx < (int)un.rows * 16; idx += nth) {
                const int r = idx >> 4, k = idx & 15;
                const float v = r < N ? a.b[un.layer][r] : 0.0f;
                __half hv = __float2half_rn(v);
                if (k == 1) hv = a.p.split ? __float2half_rn(v - __half2float(hv)) : __float2half_rn(0.0f);
                if (k > 1) hv = __float2half_rn(0.0f);
                *reinterpret_cast<__half*>(a.img + un.off + (size_t)(r >> 3) * 256 + (size_t)(k >> 3) * 128 + (size_t)(r & 7) * 16 + (k & 7) * 2) = hv;
            }
            continue;
        }
        const bool compact = un.ksteps == 1;      // a single K = 16 step: [rows / 8][2 k-chunks][8 rows][16 B], no swizzle (a quarter of the slab)
        for (int idx = tid; idx < (int)un.rows * (compact ? 16 : 64); idx += nth) {
            const int r = compact ? idx >> 4 : idx >> 6, k = compact ? idx & 15 : idx & 63;
            float v = 0.0f;
            if (un.kind < 2) {              // forward: B[n = out feature r][k = in feature]
                const int kg = un.slab * 64 + k;
                if (kg < K && r < N) v = W[(size_t)kg * N + r];
            } else {                        // backward: B[n = in feature r][k = out feature]
                const int jg = un.slab * 64 + k;
                if (r < K && jg < N) v = W[(size_t)r * N + jg];
            }
            __half hv = __float2half_rn(v);
            if (un.kind == 1) hv = __float2half_rn(v - __half2float(hv));
            const size_t eo = compact ? (size_t)(r >> 3) * 256 + (size_t)(k >> 3) * 128 + (size_t)(r & 7) * 16 + (k & 7) * 2
                                      : (size_t)r * 128 + (size_t)((((k >> 3) ^ (r & 7))) << 4) + (k & 7) * 2;
            *reinterpret_cast<__half*>(a.img + un.off + eo) = hv;
        }
    }
}


// ------------------------------------------------------------------------------------------------ compile-time MMA program
// The MMA warp's scalar instruction stream is the critical path of gen_mlp_kernel: issuing NO tcgen05.mma at all leaves the kernel
// time unchanged, and ncu's source view shows ~2,500 instructions per tile in the table-driven loop for 67 MMA / commit
// instructions.  For a network known at compile time (SpecProg) the whole per-tile program is unrolled from constants: no table
// reads, no branching on unit kinds, descriptor offsets as immediates.
struct MmaCtx {
    uint32_t sA, sW, tmem_base, w_full0, w_empty0, bar_io, bar_slab0, bar_acc_e, bar_acc_h, ones_lo;
    uint32_t U, nio, spar, slot, wb_base;
    bool leader;
};
template <class SP, int G, int U, int UEND>
struct UnitSeq {
    static __device__ __forceinline__ void run(MmaCtx& c, uint8_t* img_dst) {
        constexpr GGemm gm = SP::P.gemm[G];
        constexpr uint32_t r = SP::P.rec[U];
        constexpr uint32_t ks = (r >> 16) & 7u, kind = (r >> 19) & 3u, slab = (r >> 24) & 7u;
        constexpr uint32_t idesc = idesc_f16(TC_M, gm.N);
        constexpr uint32_t HI_SW = 0x40004040u, HI_NOSW = 0x4010u, HI_ONES = 0x4000u;
        constexpr uint32_t acc0 = U == gm.u0 ? 0u : 1u;
        if constexpr ((r & GR_SLABWAIT) != 0) {
            mbar_wait_or_trap(c.bar_slab0 + 8u * slab, (c.spar >> slab) & 1u);
            c.spar ^= 1u << slab;
            tc_fence_after();
        }
        if constexpr ((r & GR_STORE) != 0) {
            if (c.leader) {
                g_bulk_store(img_dst + (size_t)slab * GN_SLAB, c.sA + slab * GN_SLAB, GN_SLAB);
                bulk_commit();
            }
        }
        if constexpr ((r & GR_FIRST) != 0) {
            c.slot = c.U % GN_NSLOT;
            mbar_wait_or_trap(c.w_full0 + 8u * c.slot, (c.U / GN_NSLOT) & 1u);
            c.wb_base = (c.sW + c.slot * GN_SLOT) >> 4;
        }
        if (c.leader) {
            const uint32_t dcol = c.tmem_base + (uint32_t)(G & 1) * 256u;
            const uint32_t wb_lo = c.wb_base + (r & 0xFFFFu);
            const uint32_t b_ns = wb_lo | (8u << 16), b_lo = wb_lo | (1u << 16);
            const uint32_t a_lo = ((c.sA >> 4) | (1u << 16)) + slab * (uint32_t)(GN_SLAB >> 4);
            const uint32_t a_l2 = a_lo + (uint32_t)(4 * GN_SLAB >> 4);
            if constexpr (kind == 3) {
                umma_w(dcol, c.ones_lo, HI_ONES, b_ns, HI_NOSW, idesc, acc0);
            } else if constexpr (ks == 1) {
                umma_w(dcol, a_lo, HI_SW, b_ns, HI_NOSW, idesc, acc0);
                if constexpr ((r & GR_LOPART) != 0) umma_w(dcol, a_l2, HI_SW, b_ns, HI_NOSW, idesc, 1u);
            } else {
#pragma unroll
                for (uint32_t q = 0; q < ks; ++q) umma_w(dcol, a_lo + 2u * q, HI_SW, b_lo + 2u * q, HI_SW, idesc, q ? 1u : acc0);
                if constexpr ((r & GR_LOPART) != 0) {
#pragma unroll
                    for (uint32_t q = 0; q < ks; ++q) umma_w(dcol, a_l2 + 2u * q, HI_SW, b_lo + 2u * q, HI_SW, idesc, 1u);
                }
            }
            if constexpr ((r & GR_LAST) != 0) umma_commit(c.w_empty0 + 8u * c.slot);
        }
        if constexpr ((r & GR_LAST) != 0) ++c.U;
        UnitSeq<SP, G, U + 1, UEND>::run(c, img_dst);
    }
};
template <class SP, int G, int UEND>
struct UnitSeq<SP, G, UEND, UEND> {
    static __device__ __forceinline__ void run(MmaCtx&, uint8_t*) {}
};
template <class SP, int G, int GEND>
struct GemmSeq {
    static __device__ __forceinline__ void run(MmaCtx& c, const GenArgs& a, int64_t tile) {
        constexpr GGemm gm = SP::P.gemm[G];
        constexpr bool store = SP::P.fb != 0 && G > 0;
        if constexpr (gm.from_io != 0) {
            mbar_wait_or_trap(c.bar_io, c.nio & 1u); ++c.nio;
            tc_fence_after();
        }
        uint8_t* img_dst = nullptr;
        if constexpr (store) {
            constexpr int nsl = !gm.bwd ? (SP::P.width[gm.layer - 1] >> 6) : (gm.layer == SP::P.L - 1 ? 1 : (SP::P.width[gm.layer] >> 6));
            img_dst = (!gm.bwd ? a.himg[gm.layer - 1] : a.dlimg[gm.layer]) + (size_t)tile * nsl * GN_SLAB;
        }
        UnitSeq<SP, G, gm.u0, gm.u0 + gm.nu>::run(c, img_dst);
        if (c.leader) {
            if constexpr (store) bulk_wait_read();
            umma_commit(gm.head ? c.bar_acc_h : c.bar_acc_e);
        }
        GemmSeq<SP, G + 1, GEND>::run(c, a, tile);
    }
};
template <class SP, int GEND>
struct GemmSeq<SP, GEND, GEND> {
    static __device__ __forceinline__ void run(MmaCtx&, const GenArgs&, int64_t) {}
};

// ------------------------------------------------------------------------------------------------ the tile kernel
// kAct: the hidden activation is a compile-time choice (the Sigmoid epilogue would cost the ReLU one registers);
// kDbg compiles the phase clocks in (B2048_DBG_TC_CLOCKS)
// kSpec != 0: the MMA warp runs the compile-time program of SpecProg<kSpec, kSplit, kFb> (the host launches it only for that network)
// kEnt (update mode, policy head): the head delta carries the entropy bonus, d_j = coef (1[a = j] - p_j) - ecoef t_j
// (b2048_entropy.cuh), and ent.ent_sum (nullable) += sum_s H_s
struct GenEnt {
    const float* ent_coef;
    double* ent_sum;
};
struct GenEntArgs {
    GenArgs g;
    GenEnt e;
};

template <int kAct, bool kDbg, int kSpec, bool kSplit, bool kFb, bool kEnt>
__device__ __forceinline__ void gen_mlp_body(const GenArgs& a, const GenEnt& ent) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + GS_BAR);
    const uint32_t w_full0 = s_u32(&bars[0]), w_empty0 = s_u32(&bars[3]);
    const uint32_t bar_io = s_u32(&bars[6]), bar_acc_e = s_u32(&bars[8]), bar_acc_h = s_u32(&bars[9]), bar_free = s_u32(&bars[10]);
    const uint32_t bar_slab0 = s_u32(&bars[11]);   // [11..14] slab s of the A operand written by the epilogue warps
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + GS_BAR + 128);
    const GenProg& P = a.p;

    if (tid == 0) {
        for (int i = 0; i < GN_NSLOT; ++i) { mbar_init(w_full0 + 8u * i, 1); mbar_init(w_empty0 + 8u * i, 1); }
        mbar_init(bar_io, 4);        // the I/O warps have written an A operand (the tile's input; its head deltas)
        for (int i = 0; i < 4; ++i) mbar_init(bar_slab0 + 8u * i, 16);   // the epilogue warps have written slab i of an A operand
        mbar_init(bar_acc_e, 1);     // an accumulator for the epilogue warps is complete
        mbar_init(bar_acc_h, 1);     // the head accumulator (I/O warps) is complete
        mbar_init(bar_free, 1);      // update mode: the tile's last image has left the A buffer
        mbar_init_fence();
    }
    if (tid < 64) {      // ONES operand: [2 k-chunks][8 rows][8 halves]; chunk 0 of every row = (1, 1, 0, ...)
        const int e = tid & 7, chunk = tid >> 5;
        reinterpret_cast<uint32_t*>(smem + GS_ONES)[tid] = 0u;
        if (chunk == 0 && (e & 3) == 0) reinterpret_cast<uint32_t*>(smem + GS_ONES)[tid] = 0x3C003C00u;
        fence_proxy_async_smem();
    }
    const uint32_t tmem_base = tmem_setup(warp == 16, tmem_slot, 512u);
    const int64_t n_eff = a.n_dev ? (int64_t)*a.n_dev : a.n;        // uniform over the grid
    const int64_t n_tiles = (n_eff + TC_M - 1) / TC_M;
    const uint32_t sA = s_u32(smem + GS_A), sW = s_u32(smem + GS_W);

    if (warp == 16) {
        // ============================ MMA warp: GEMM program, image stores ============================
        // A GEMM whose A operand comes from the epilogue warps starts on K slab s as soon as THAT slab has been written (per-slab
        // barriers): the epilogue of GEMM G runs under the MMAs of GEMM G + 1 (accumulators alternate between two TMEM regions).
        // All 32 lanes walk the program CONVERGENTLY (loop counters, table reads and descriptor words stay in uniform registers);
        // only the asynchronous instructions themselves are issued by lane 0 (with the whole loop under `if (lane == 0)` every
        // tcgen05.mma cost ~25 vector instructions: ELECT / R2UR per operand).
        if constexpr (kSpec != 0) {
            using SP = SpecProg<kSpec, kSplit, kFb>;
            MmaCtx c;
            c.sA = sA; c.sW = sW; c.tmem_base = tmem_base; c.w_full0 = w_full0; c.w_empty0 = w_empty0; c.bar_io = bar_io;
            c.bar_slab0 = bar_slab0; c.bar_acc_e = bar_acc_e; c.bar_acc_h = bar_acc_h;
            c.ones_lo = (s_u32(smem + GS_ONES) >> 4) | (8u << 16);
            c.U = 0; c.nio = 0; c.spar = 0; c.slot = 0; c.wb_base = 0; c.leader = lane == 0;
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                GemmSeq<SP, 0, SP::P.n_gemm>::run(c, a, tile);
                if constexpr (kFb) {       // delta_0 (the last epilogue's output) is only an image
                    constexpr int nsl = SP::P.width[0] >> 6;
#pragma unroll
                    for (int sl = 0; sl < nsl; ++sl) {
                        mbar_wait_or_trap(bar_slab0 + 8u * (uint32_t)sl, (c.spar >> sl) & 1u);
                        c.spar ^= 1u << sl;
                        if (c.leader) g_bulk_store(a.dlimg[0] + ((size_t)tile * nsl + sl) * GN_SLAB, sA + (uint32_t)sl * GN_SLAB, GN_SLAB);
                    }
                    if (c.leader) {
                        bulk_commit();
                        bulk_wait_read();
                        mbar_arrive(bar_free);
                    }
                }
            }
            if (c.leader) bulk_wait();
        } else {
            const bool leader = lane == 0;
            uint32_t U = 0, nio = 0, spar = 0;      // ring fills consumed; I/O hand-offs; phase parity of the four slab barriers
            constexpr uint32_t HI_SW = 0x40004040u, HI_NOSW = 0x4010u, HI_ONES = 0x4000u;     // upper descriptor words (b2048_tc.cuh)
            const uint32_t ones_lo = (s_u32(smem + GS_ONES) >> 4) | (8u << 16);
            int lt = 0;
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++lt) {
                long long* dc = (kDbg && a.dbg && blockIdx.x == 0 && lt < 4 && leader) ? a.dbg + 64 * lt : nullptr;
                if (dc) dc[0] = clock64();
                for (int G = 0; G < P.n_gemm; ++G) {
                    const GGemm gm = P.gemm[G];
                    const bool from_io = gm.from_io != 0;
                    long long wsum = 0;
                    if (from_io) {
                        mbar_wait_or_trap(bar_io, nio & 1u); ++nio;
                        tc_fence_after();
                        if (dc) dc[1 + 3 * G] = clock64();
                    }
                    // in update mode the A operand of every GEMM but the first is an image the dW GEMMs read
                    const bool store = P.fb && G > 0;
                    uint8_t* img_dst = nullptr;
                    if (store) {
                        const int nsl = !gm.bwd ? (P.width[gm.layer - 1] >> 6) : (gm.layer == P.L - 1 ? 1 : (P.width[gm.layer] >> 6));
                        img_dst = (!gm.bwd ? a.himg[gm.layer - 1] : a.dlimg[gm.layer]) + (size_t)tile * nsl * GN_SLAB;
                    }
                    const uint32_t dcol = tmem_base + (uint32_t)(G & 1) * 256u;
                    const uint32_t idesc = idesc_f16(TC_M, gm.N);
                    uint32_t acc = 0u;
                    for (int f = gm.f0; f < gm.f0 + gm.nf; ++f, ++U) {
                        const GFill fl = P.fill[f];
                        const uint32_t slot = U % GN_NSLOT, use = U / GN_NSLOT;
                        bool loaded = false;
                        for (int u = fl.u0; u < fl.u0 + fl.nu; ++u) {
                            const GUnit un = P.unit[u];
                            if (un.kind == 0 || un.kind == 2) {      // first unit of K slab un.slab
                                if (!from_io) {
                                    mbar_wait_or_trap(bar_slab0 + 8u * (uint32_t)un.slab, (spar >> un.slab) & 1u);
                                    spar ^= 1u << un.slab;
                                    tc_fence_after();
                                    if (dc && un.slab == 0) dc[1 + 3 * G] = clock64();
                                }
                                if (store && leader) {
                                    g_bulk_store(img_dst + (size_t)un.slab * GN_SLAB, sA + (uint32_t)un.slab * GN_SLAB, GN_SLAB);
                                    bulk_commit();
                                }
                            }
                            if (!loaded) {
                                const long long w0 = dc ? clock64() : 0;
                                mbar_wait_or_trap(w_full0 + 8u * slot, use & 1u);
                                if (dc) wsum += clock64() - w0;
                                loaded = true;
                            }
                            const uint32_t wb_lo = ((sW + slot * GN_SLOT) >> 4) + (uint32_t)un.slot_off16;
                            const uint32_t a_lo = ((sA + (uint32_t)un.slab * GN_SLAB) >> 4) | (1u << 16);
                            // one divergent region per unit, straight-line inside: the warp's scalar instruction stream is the
                            // critical path of the kernel (issuing NO MMAs at all leaves the kernel time unchanged), and every
                            // branch / convergence barrier around a tcgen05.mma costs more than the instruction itself
                            if (leader) {
                                const uint32_t b_ns = wb_lo | (8u << 16), b_lo = wb_lo | (1u << 16);
                                const uint32_t a_l2 = a_lo + (uint32_t)(4 * GN_SLAB >> 4);
                                const bool lo_part = un.kind == 0 && gm.a_lo;
                                if (un.kind == 3) {                  // bias: constant ones A operand, [N x 16] no-swizzle B
                                    umma_w(dcol, ones_lo, HI_ONES, b_ns, HI_NOSW, idesc, acc);
                                } else if (un.ksteps == 4) {
                                    umma_w(dcol, a_lo, HI_SW, b_lo, HI_SW, idesc, acc);
                                    umma_w(dcol, a_lo + 2u, HI_SW, b_lo + 2u, HI_SW, idesc, 1u);
                                    umma_w(dcol, a_lo + 4u, HI_SW, b_lo + 4u, HI_SW, idesc, 1u);
                                    umma_w(dcol, a_lo + 6u, HI_SW, b_lo + 6u, HI_SW, idesc, 1u);
                                    if (lo_part) {
                                        umma_w(dcol, a_l2, HI_SW, b_lo, HI_SW, idesc, 1u);
                                        umma_w(dcol, a_l2 + 2u, HI_SW, b_lo + 2u, HI_SW, idesc, 1u);
                                        umma_w(dcol, a_l2 + 4u, HI_SW, b_lo + 4u, HI_SW, idesc, 1u);
                                        umma_w(dcol, a_l2 + 6u, HI_SW, b_lo + 6u, HI_SW, idesc, 1u);
                                    }
                                } else if (un.ksteps == 1) {         // compact single-K-step unit (no-swizzle B)
                                    umma_w(dcol, a_lo, HI_SW, b_ns, HI_NOSW, idesc, acc);
                                    if (lo_part) umma_w(dcol, a_l2, HI_SW, b_ns, HI_NOSW, idesc, 1u);
                                } else {                             // 2 or 3 K steps (an input width that is not a multiple of 64)
                                    for (uint32_t q = 0; q < un.ksteps; ++q) umma_w(dcol, a_lo + 2u * q, HI_SW, b_lo + 2u * q, HI_SW, idesc, q ? 1u : acc);
                                    if (lo_part)
                                        for (uint32_t q = 0; q < un.ksteps; ++q) umma_w(dcol, a_l2 + 2u * q, HI_SW, b_lo + 2u * q, HI_SW, idesc, 1u);
                                }
                            }
                            acc = 1u;
                        }
                        if (leader) umma_commit(w_empty0 + 8u * slot);
                    }
                    // the epilogue of this GEMM overwrites the A buffer: the image stores must have read it
                    if (store && leader) bulk_wait_read();
                    if (leader) umma_commit(gm.head ? bar_acc_h : bar_acc_e);
                    if (dc) { dc[2 + 3 * G] = clock64(); dc[3 + 3 * G] = wsum; }
                }
                if (P.fb) {            // delta_0 (the last epilogue's output) is only an image
                    const int nsl = P.width[0] >> 6;
                    for (int sl = 0; sl < nsl; ++sl) {
                        mbar_wait_or_trap(bar_slab0 + 8u * (uint32_t)sl, (spar >> sl) & 1u);
                        spar ^= 1u << sl;
                        if (leader) g_bulk_store(a.dlimg[0] + ((size_t)tile * nsl + sl) * GN_SLAB, sA + (uint32_t)sl * GN_SLAB, GN_SLAB);
                    }
                    if (leader) {
                        bulk_commit();
                        bulk_wait_read();
                        mbar_arrive(bar_free);
                    }
                }
            }
            if (leader) bulk_wait();
        }
        __syncwarp();
    } else if (warp == 17) {
        // ============================ weight loader ============================
        if (lane == 0) {
            uint32_t U = 0;
            for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                for (int f = 0; f < P.n_fills; ++f, ++U) {
                    const GFill fl = P.fill[f];
                    const uint32_t slot = U % GN_NSLOT, use = U / GN_NSLOT;
                    if (use > 0) mbar_wait_or_trap(w_empty0 + 8u * slot, (use - 1u) & 1u);
                    const uint32_t bar = w_full0 + 8u * slot, bytes = (uint32_t)fl.bytes16 * 16u;
                    mbar_expect_tx(bar, bytes);
                    bulk_load_chunked<16384u>(sW + slot * GN_SLOT, a.img + fl.off, bytes, bar);
                }
            }
        }
        __syncwarp();
    } else if (warp < 16) {
        // ============================ epilogue warps: accumulator -> next A operand ============================
        // (biases arrive through the bias MMA; mask bit of column i of a 16-column group sits at bit 15 - i)
        const int q = warp & 3, g = warp >> 2;
        const int row = q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        uint16_t* msk = a.mask_scratch ? a.mask_scratch + (size_t)blockIdx.x * GN_MASK_WORDS : nullptr;
        uint4* dsg = a.dsig_scratch ? a.dsig_scratch + (size_t)blockIdx.x * GN_MASK_WORDS * 2 : nullptr;
        uint8_t* a_row = smem + GS_A + row * 128;
        uint32_t ne = 0;
        int lt = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++lt) {
            long long* dc = (kDbg && a.dbg && blockIdx.x == 0 && tid == 0 && lt < 4) ? a.dbg + 64 * lt : nullptr;
            for (int G = 0; G < P.n_gemm; ++G) {
                const GGemm gm = P.gemm[G];
                if (gm.head) continue;
                mbar_wait_or_trap(bar_acc_e, ne & 1u); ++ne;
                if (dc) dc[32 + 2 * G] = clock64();
                tc_fence_after();
                const uint32_t dcol = tlane + (uint32_t)(G & 1) * 256u + (uint32_t)(g * 16);
                const int nsl = gm.N >> 6;
                uint32_t r[2][16];
                tmem_ld16_issue(dcol, r[0]);                 // the TMEM load of slab s + 1 is in flight while slab s is converted
#pragma unroll
                for (int s = 0; s < 4; ++s) {
                    if (s >= nsl) break;
                    uint32_t (&rc)[16] = r[s & 1];
                    tmem_ld_wait(rc);
                    if (s + 1 < nsl) tmem_ld16_issue(dcol + (uint32_t)((s + 1) * 64), r[(s + 1) & 1]);
                    if (!gm.bwd && kAct == B2048_ACTV_SIGMOID) {
                        // a = 1 / (1 + exp(-z)) (MLP.py:132); the update keeps s (1 - s) for the backward pass
                        uint32_t dg[8];
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            uint32_t hi[4], lo[4];
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const float s0 = 1.0f / (1.0f + expf(-__uint_as_float(rc[8 * c + 2 * k])));
                                const float s1 = 1.0f / (1.0f + expf(-__uint_as_float(rc[8 * c + 2 * k + 1])));
                                hi[k] = pack_f16(s0, s1);
                                const float2 hf = __half22float2(*reinterpret_cast<__half2*>(&hi[k]));
                                lo[k] = pack_f16(s0 - hf.x, s1 - hf.y);
                                dg[4 * c + k] = pack_f16(s0 * (1.0f - s0), s1 * (1.0f - s1));
                            }
                            const int sw = ((g * 2 + c) ^ (row & 7)) << 4;
                            *reinterpret_cast<uint4*>(a_row + s * GN_SLAB + sw) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                            if (P.split) *reinterpret_cast<uint4*>(a_row + (4 + s) * GN_SLAB + sw) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                        }
                        if (dsg) {
                            uint4* d = dsg + (size_t)(((gm.layer * 4 + s) * 4 + g) * 128 + row) * 2;
                            d[0] = make_uint4(dg[0], dg[1], dg[2], dg[3]);
                            d[1] = make_uint4(dg[4], dg[5], dg[6], dg[7]);
                        }
                    } else if (gm.bwd && kAct == B2048_ACTV_SIGMOID) {
                        // delta_{layer-1} = D . s (1 - s)
                        const uint4* d = dsg + (size_t)((((gm.layer - 1) * 4 + s) * 4 + g) * 128 + row) * 2;
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            const uint4 dv = d[c];
                            const uint32_t dw[4] = {dv.x, dv.y, dv.z, dv.w};
                            uint32_t o[4];
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const float2 df = __half22float2(*reinterpret_cast<const __half2*>(&dw[k]));
                                o[k] = pack_f16(__uint_as_float(rc[8 * c + 2 * k]) * df.x, __uint_as_float(rc[8 * c + 2 * k + 1]) * df.y);
                            }
                            const int sw = ((g * 2 + c) ^ (row & 7)) << 4;
                            *reinterpret_cast<uint4*>(a_row + s * GN_SLAB + sw) = make_uint4(o[0], o[1], o[2], o[3]);
                        }
                    } else if (!gm.bwd) {
                        uint32_t m = 0;
#pragma unroll
                        for (int i = 0; i < 16; ++i) m = __funnelshift_l(0u - rc[i], m, 1);     // z > 0  <=>  sign bit of -bits(z)
                        if (msk) msk[((gm.layer * 4 + s) * 4 + g) * 128 + row] = (uint16_t)m;
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            uint32_t hi[4], lo[4];
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const uint32_t b0 = rc[8 * c + 2 * k], b1 = rc[8 * c + 2 * k + 1];
                                hi[k] = relu_pack_f16(b0, b1);
                                if (P.split) {
                                    const float2 hf = __half22float2(*reinterpret_cast<__half2*>(&hi[k]));
                                    lo[k] = pack_f16(fmaxf(__uint_as_float(b0), 0.0f) - hf.x, fmaxf(__uint_as_float(b1), 0.0f) - hf.y);
                                }
                            }
                            const int sw = ((g * 2 + c) ^ (row & 7)) << 4;
                            *reinterpret_cast<uint4*>(a_row + s * GN_SLAB + sw) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
                            if (P.split) *reinterpret_cast<uint4*>(a_row + (4 + s) * GN_SLAB + sw) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
                        }
                    } else {
                        // delta_{layer-1} = D . [z_{layer-1} > 0]
                        const uint32_t m = msk[(((gm.layer - 1) * 4 + s) * 4 + g) * 128 + row];
#pragma unroll
                        for (int c = 0; c < 2; ++c) {
                            uint32_t o[4];
#pragma unroll
                            for (int k = 0; k < 4; ++k) {
                                const int i0 = 8 * c + 2 * k;
                                const float x0 = (m >> (15 - i0)) & 1u ? __uint_as_float(rc[i0]) : 0.0f;
                                const float x1 = (m >> (14 - i0)) & 1u ? __uint_as_float(rc[i0 + 1]) : 0.0f;
                                o[k] = pack_f16(x0, x1);
                            }
                            const int sw = ((g * 2 + c) ^ (row & 7)) << 4;
                            *reinterpret_cast<uint4*>(a_row + s * GN_SLAB + sw) = make_uint4(o[0], o[1], o[2], o[3]);
                        }
                    }
                    fence_proxy_async_smem();
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(bar_slab0 + 8u * (uint32_t)s);
                }
                if (dc) dc[33 + 2 * G] = clock64();
            }
        }
    } else {
        // ============================ I/O warps (18..21), one thread per sample ============================
        const int q = warp & 3;             // a TMEM load may only touch the lane quarter warp % 4
        const int row = q * 32 + lane;
        const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
        const uint32_t hcol = (uint32_t)((P.L - 1) & 1) * 256u;     // the head GEMM is GEMM L - 1
        const float* bh = a.bias[P.L - 1];
        float b4[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) b4[j] = j < P.n_out ? __ldg(bh + j) : 0.0f;
        const float S = P.fb ? a.scale[0] : 1.0f;
        const bool use_mask = a.mask_flags != nullptr;
        uint32_t lt = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++lt) {
            long long* dc = (kDbg && a.dbg && blockIdx.x == 0 && warp == 18 && lane == 0 && lt < 4) ? a.dbg + 64 * lt : nullptr;
            if (dc) dc[60] = clock64();
            const int64_t slot = tile * TC_M + row;
            const bool valid = slot < n_eff;
            const int64_t s = (valid && a.slot_map) ? (int64_t)a.slot_map[slot] : slot;     // the board behind the slot
            const uint64_t bd = valid ? a.board[s] : 0ull;
            uint32_t fl = 0xFu, act = 0u;
            float cf = 0.0f, ecf = 0.0f;
            if (valid) {
                if (use_mask) fl = a.mask_flags[s];
                if (P.fb) { cf = a.coef[s]; if (a.act_in) act = a.act_in[s]; }
                if constexpr (kEnt) ecf = ent.ent_coef[s];
            }
            uint32_t w3 = 0u;
            if (valid && !P.fb && a.action && !a.greedy) w3 = stream_keyed(a.keys, a.gid0 + (uint64_t)s, a.t, B2048_DOM_STEP).w3;
            // the A buffer is free: forward-only, the previous tile's head GEMM has completed (waited for below); update mode,
            // its last image has been read out
            if (P.fb && lt > 0) mbar_wait_or_trap(bar_free, (lt - 1u) & 1u);
            if (dc) dc[61] = clock64();
            if (P.obs_mode == B2048_OBS_ONEHOT) {
                zero_slabs_128(smem + GS_A, P.in_slabs, tid - 18 * 32);
                bar_sync(1, 128);                     // the four I/O warps only
            }
            encode_input_row(bd, row, smem + GS_A, 0, P.in_slabs, P.obs_mode, P.obs_scale);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_io);
            if (dc) dc[62] = clock64();
            mbar_wait_or_trap(bar_acc_h, lt & 1u);
            if (dc) dc[63] = clock64();
            tc_fence_after();
            uint32_t r4[4];
            tmem_ld4(tlane + hcol, r4);
            tc_fence_before();
            float lg[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) lg[j] = __uint_as_float(r4[j]) + b4[j];
            float p[4] = {0.0f, 0.0f, 0.0f, 0.0f};
            float ent_t[4] = {0.0f, 0.0f, 0.0f, 0.0f}, ent_h = 0.0f;
            if (!P.fb || a.head_mode == 0) {
                float m[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) m[j] = (j >= P.n_out) ? -INFINITY : ((use_mask && !((fl >> j) & 1u)) ? -1e9f : lg[j]);   // MLP.py:144-146
                const float mx = fmaxf(fmaxf(m[0], m[1]), fmaxf(m[2], m[3]));
                float sum = 0.0f;
#pragma unroll
                for (int j = 0; j < 4; ++j) { p[j] = expf(m[j] - mx); sum += p[j]; }
                const float inv = 1.0f / sum;
#pragma unroll
                for (int j = 0; j < 4; ++j) p[j] *= inv;
                if constexpr (kEnt) {
                    float z[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j) z[j] = m[j] - mx;
                    ent_h = entropy_row(z, logf(sum), p, use_mask ? fl : 0xFu, P.n_out, ent_t);
                }
            }
            if (!P.fb) {
                if (valid) {
                    for (int j = 0; j < P.n_out; ++j) {
                        if (a.out) a.out[s * P.n_out + j] = lg[j];
                        if (a.logits) a.logits[s * P.n_out + j] = lg[j];
                        if (a.probs) a.probs[s * P.n_out + j] = p[j];
                    }
                    if (a.action) {
                        uint32_t ac = 0;
                        if (a.greedy) {      // int(np.argmax(probs * mask)): first maximum wins (reinforce_agent.py:179-185)
                            float best = -1.0f;
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const float qj = (j < P.n_out && (!use_mask || ((fl >> j) & 1u))) ? p[j] : (j < P.n_out ? 0.0f : -1.0f);
                                if (qj > best) { best = qj; ac = (uint32_t)j; }
                            }
                        } else {             // rng.choice(4, p=probs) as an inverse CDF on the board's Philox word 3 (reinforce_agent.py:187)
                            const float c0 = p[0], c1 = c0 + p[1], c2 = c1 + p[2], c3 = c2 + p[3];
                            const float u = ((float)(w3 >> 8) + 0.5f) * (1.0f / 16777216.0f) * c3;
                            ac = (u >= c0 ? 1u : 0u) + (u >= c1 ? 1u : 0u) + (u >= c2 ? 1u : 0u);
                            if (!(p[ac] > 0.0f)) {
                                if (p[3] > 0.0f) ac = 3;
                                if (p[2] > 0.0f) ac = 2;
                                if (p[1] > 0.0f) ac = 1;
                                if (p[0] > 0.0f) ac = 0;
                            }
                        }
                        a.action[s] = (uint8_t)ac;
                    }
                }
            } else {
                float d[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                if (a.head_mode == 0) {
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        if (j < P.n_out) {
                            if constexpr (kEnt) d[j] = cf * ((act == (uint32_t)j ? 1.0f : 0.0f) - p[j]) - ecf * ent_t[j];
                            else d[j] = cf * ((act == (uint32_t)j ? 1.0f : 0.0f) - p[j]);     // reinforce_agent.py:340-344
                        }
                    if constexpr (kEnt) {
                        if (ent.ent_sum) {                                                            // one float64 atomic per warp and tile
                            float hs = valid ? ent_h : 0.0f;
#pragma unroll
                            for (int o = 16; o > 0; o >>= 1) hs += __shfl_xor_sync(0xFFFFFFFFu, hs, o);
                            if (lane == 0 && hs != 0.0f) atomicAdd(ent.ent_sum, (double)hs);
                        }
                    }
                } else {
                    d[0] = cf;                                                                        // dLoss/dV * weight
                }
                // head deltas as the fp16 A operand of the first backward GEMM (K = 16: chunks 0 and 1 of slab 0) — the head GEMM has
                // completed, so the A buffer is free
                uint8_t* a_row = smem + GS_A + row * 128;
                const int sw = row & 7;
                *reinterpret_cast<uint4*>(a_row + ((0 ^ sw) << 4)) = make_uint4(pack_f16(d[0] * S, d[1] * S), pack_f16(d[2] * S, d[3] * S), 0u, 0u);
                *reinterpret_cast<uint4*>(a_row + ((1 ^ sw) << 4)) = make_uint4(0u, 0u, 0u, 0u);
                fence_proxy_async_smem();
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_io);
                // head bias gradient (unscaled float32 sum over the warp's 32 samples)
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    float v = d[j];
#pragma unroll
                    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xFFFFFFFFu, v, o);
                    if (lane == 0 && j < P.n_out && v != 0.0f) atomicAdd(a.gb_head + j, v);
                }
            }
            if (dc) dc[59] = clock64();
        }
    }

    tmem_teardown(warp == 16, tmem_base, 512u);
}

template <int kAct, bool kDbg, int kSpec, bool kSplit, bool kFb>
__global__ void __launch_bounds__(GN_THREADS, 1) gen_mlp_kernel(const __grid_constant__ GenArgs a) {
    gen_mlp_body<kAct, kDbg, kSpec, kSplit, kFb, false>(a, GenEnt{});
}

// update mode with the entropy bonus in the policy head's delta
template <int kAct, int kSpec, bool kSplit, bool kFb>
__global__ void __launch_bounds__(GN_THREADS, 1) gen_mlp_ent_kernel(const __grid_constant__ GenEntArgs a) {
    gen_mlp_body<kAct, false, kSpec, kSplit, kFb, true>(a.g, a.e);
}

// ------------------------------------------------------------------------------------------------ dW GEMMs
struct GenDwArgs {
    const uint8_t* aimg;       // activation image of the layer's input, or NULL: regenerated from the boards (layer 0)
    const uint64_t* board;
    int obs_mode;
    float obs_scale;
    const uint8_t* bimg;       // delta image of the layer
    int a_slabs, b_slabs;      // slabs per tile of the two images
    int N;                     // MMA N: the layer's width (head: 16)
    int K_real, N_real;        // dW is [K_real][N_real] row-major
    float* gW;
    float* gb;                 // nullable (head: accumulated by gen_mlp_kernel)
    const float* inv_scale;
    int64_t n_tiles, n;
    int mtiles, ksplit, stages;
    uint32_t tmem_cols;
};
constexpr int GD_THREADS = 10 * 32;    // loader, MMA, 4 column-sum / read-out warps, 4 input-generator warps

__global__ void __launch_bounds__(GD_THREADS, 1) gen_dw_kernel(const __grid_constant__ GenDwArgs a) {
    extern __shared__ __align__(1024) uint8_t smem[];
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int stage_bytes = 2 * GN_SLAB + a.b_slabs * GN_SLAB;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + a.stages * stage_bytes);
    const uint32_t full0 = s_u32(&bars[0]), empty0 = s_u32(&bars[4]), bar_done = s_u32(&bars[8]);
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + a.stages * stage_bytes + 128);
    const int mt = (int)blockIdx.x % a.mtiles, ks = (int)blockIdx.x / a.mtiles;
    const bool gen = a.aimg == nullptr;
    const int a_have = a.a_slabs - 2 * mt < 2 ? a.a_slabs - 2 * mt : 2;
    const int ncs = (mt == 0 && a.gb != nullptr) ? a.b_slabs : 0;      // column-sum warps (bias gradient) of this CTA
    if (tid == 0) {
        for (int i = 0; i < a.stages; ++i) { mbar_init(full0 + 8u * i, gen ? 5 : 1); mbar_init(empty0 + 8u * i, 1 + ncs); }
        mbar_init(bar_done, 1);
        mbar_init_fence();
    }
    // a missing second A slab (a 64- or 272-feature input) stays zero for the whole kernel
    for (int i = tid; i < a.stages * 2 * GN_SLAB / 16; i += GD_THREADS) {
        const int st = i / (2 * GN_SLAB / 16), o = i % (2 * GN_SLAB / 16);
        *reinterpret_cast<uint4*>(smem + st * stage_bytes + o * 16) = make_uint4(0u, 0u, 0u, 0u);
    }
    fence_proxy_async_smem();
    const uint32_t tmem_base = tmem_setup(warp == 1, tmem_slot, a.tmem_cols);
    const int64_t n_my = ks < a.n_tiles ? (a.n_tiles - ks + a.ksplit - 1) / a.ksplit : 0;

    if (warp == 0) {
        if (lane == 0) {
            for (int64_t it = 0; it < n_my; ++it) {
                const int st = (int)(it % a.stages);
                const int64_t use = it / a.stages, tile = ks + it * a.ksplit;
                if (use > 0) mbar_wait_or_trap(empty0 + 8u * st, (uint32_t)(use - 1) & 1u);
                const uint32_t bar = full0 + 8u * st;
                const uint32_t ab = gen ? 0u : (uint32_t)(a_have * GN_SLAB), bb = (uint32_t)(a.b_slabs * GN_SLAB);
                mbar_expect_tx(bar, ab + bb);
                const uint32_t sa = s_u32(smem + st * stage_bytes);
                if (!gen) bulk_load_chunked<16384u>(sa, a.aimg + ((size_t)tile * a.a_slabs + 2 * mt) * GN_SLAB, ab, bar);
                bulk_load_chunked<16384u>(sa + 2u * GN_SLAB, a.bimg + (size_t)tile * a.b_slabs * GN_SLAB, bb, bar);
            }
        }
        __syncwarp();
    } else if (warp == 1) {
        if (lane == 0) {
            const uint32_t idesc = idesc_f16(128, a.N) | kIdescAMn | kIdescBMn;
            for (int64_t it = 0; it < n_my; ++it) {
                const int st = (int)(it % a.stages);
                mbar_wait_or_trap(full0 + 8u * st, (uint32_t)(it / a.stages) & 1u);
                tc_fence_after();
                const uint32_t sa = s_u32(smem + st * stage_bytes), sb = sa + 2u * GN_SLAB;
#pragma unroll
                for (int kk = 0; kk < 8; ++kk)            // 16 samples per MMA; M = 128 features = two slabs, N = a.N
                    umma_f16(tmem_base, desc_sw128_mn(sa + (uint32_t)kk * 2048u, GN_SLAB), desc_sw128_mn(sb + (uint32_t)kk * 2048u, GN_SLAB),
                             idesc, (it | kk) ? 1u : 0u);
                umma_commit(empty0 + 8u * st);
            }
            umma_commit(bar_done);
        }
        __syncwarp();
    } else if (warp < 6) {
        // ---- bias gradient: column sums of the staged delta image (CTAs of M tile 0), then the accumulator read-out
        const int cw = warp - 2, chunk = lane & 7, rsub = lane >> 3;
        const float inv = *a.inv_scale;
        if (cw < ncs) {
            float acc[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) acc[e] = 0.0f;
            for (int64_t it = 0; it < n_my; ++it) {
                const int st = (int)(it % a.stages);
                mbar_wait_or_trap(full0 + 8u * st, (uint32_t)(it / a.stages) & 1u);
                const uint8_t* x = smem + st * stage_bytes + 2 * GN_SLAB + cw * GN_SLAB;
#pragma unroll 4
                for (int r = rsub; r < 128; r += 4) {
                    const uint4 v = *reinterpret_cast<const uint4*>(x + r * 128 + ((chunk ^ (r & 7)) << 4));
                    const float2 f0 = __half22float2(*reinterpret_cast<const __half2*>(&v.x)), f1 = __half22float2(*reinterpret_cast<const __half2*>(&v.y));
                    const float2 f2 = __half22float2(*reinterpret_cast<const __half2*>(&v.z)), f3 = __half22float2(*reinterpret_cast<const __half2*>(&v.w));
                    acc[0] += f0.x; acc[1] += f0.y; acc[2] += f1.x; acc[3] += f1.y; acc[4] += f2.x; acc[5] += f2.y; acc[6] += f3.x; acc[7] += f3.y;
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(empty0 + 8u * st);
            }
#pragma unroll
            for (int e = 0; e < 8; ++e) {
                acc[e] += __shfl_xor_sync(0xFFFFFFFFu, acc[e], 8);
                acc[e] += __shfl_xor_sync(0xFFFFFFFFu, acc[e], 16);
            }
            if (lane < 8 && n_my > 0) {
#pragma unroll
                for (int e = 0; e < 8; ++e) {
                    const int c = cw * 64 + chunk * 8 + e;
                    if (c < a.N_real && acc[e] != 0.0f) atomicAdd(a.gb + c, acc[e] * inv);
                }
            }
        }
        if (n_my > 0) {
            mbar_wait_or_trap(bar_done, 0);
            tc_fence_after();
            const int q = warp & 3;
            const uint32_t tlane = tmem_base + ((uint32_t)(q * 32) << 16);
            const int m = mt * 128 + q * 32 + lane;                    // input feature
            const bool vec4 = (a.N_real & 3) == 0 && (reinterpret_cast<uintptr_t>(a.gW) & 15) == 0;
            for (int c0 = 0; c0 < a.N; c0 += 16) {
                uint32_t r[16];
                tmem_ld16(tlane + (uint32_t)c0, r);
                if (m < a.K_real) {
                    float* dst = a.gW + (size_t)m * a.N_real + c0;
                    if (vec4 && c0 + 16 <= a.N_real) {          // four 128-bit reductions instead of 16 scalar atomics
#pragma unroll
                        for (int i = 0; i < 16; i += 4)
                            red_add_v4(dst + i, __uint_as_float(r[i]) * inv, __uint_as_float(r[i + 1]) * inv, __uint_as_float(r[i + 2]) * inv, __uint_as_float(r[i + 3]) * inv);
                    } else {
#pragma unroll
                        for (int i = 0; i < 16; ++i) {
                            const float v = __uint_as_float(r[i]) * inv;
                            if (c0 + i < a.N_real && v != 0.0f) atomicAdd(dst + i, v);
                        }
                    }
                }
            }
        }
    } else if (gen) {
        // ---- layer 0: the input rows of the tile, regenerated from the packed boards (M tile mt = slabs 2 mt, 2 mt + 1)
        const int row = (warp - 6) * 32 + lane;
        for (int64_t it = 0; it < n_my; ++it) {
            const int st = (int)(it % a.stages);
            const int64_t use = it / a.stages, tile = ks + it * a.ksplit;
            const int64_t s = tile * 128 + row;
            const uint64_t bd = s < a.n ? a.board[s] : 0ull;
            if (use > 0) mbar_wait_or_trap(empty0 + 8u * st, (uint32_t)(use - 1) & 1u);
            if (a.obs_mode == B2048_OBS_ONEHOT) {
                zero_slabs_128(smem + st * stage_bytes, a_have, tid - 6 * 32);
                bar_sync(2, 128);                     // the four generator warps only
            }
            encode_input_row(bd, row, smem + st * stage_bytes, 2 * mt, a_have, a.obs_mode, a.obs_scale);
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) mbar_arrive(full0 + 8u * st);
        }
    }
    // written out: tmem_teardown() would load a.tmem_cols ahead of the branch and change the SASS
    tc_fence_before();
    __syncthreads();
    if (warp == 1) tmem_dealloc(tmem_base, a.tmem_cols);
}

// ------------------------------------------------------------------------------------------------ host side
// Shapes: 1..4 hidden layers whose sizes are multiples of 64 up to 256, ReLU or Sigmoid, log2 (16-wide) or one-hot (272-wide)
// input, 1..4 outputs.  (Raw observations reach 32768 per input and could leave the fp16 range in the activations.)
bool gen_shape_ok(const b2048_mlp_desc* mlp) {
    if (!mlp || mlp->n_layers < 2 || mlp->n_layers > GN_MAXL) return false;
    if (mlp->activation != B2048_ACTV_RELU && mlp->activation != B2048_ACTV_SIGMOID) return false;
    if (!((mlp->obs_mode == B2048_OBS_LOG2 && mlp->dims[0] == 16) || (mlp->obs_mode == B2048_OBS_ONEHOT && mlp->dims[0] == 272))) return false;
    for (int l = 1; l < mlp->n_layers; ++l)
        if (mlp->dims[l] < 64 || mlp->dims[l] > 256 || mlp->dims[l] % 64 != 0) return false;
    const int n_out = mlp->dims[mlp->n_layers];
    if (n_out < 1 || n_out > 4) return false;
    for (int l = 0; l < mlp->n_layers; ++l)
        if (!mlp->W[l] || !mlp->b[l]) return false;
    return true;
}
bool gen_supported(const b2048_handle* h, const b2048_mlp_desc* mlp) { return gen_shape_ok(mlp) && h->smem_optin >= 227 * 1024; }

static void build_program(const b2048_mlp_desc* mlp, bool split, bool fb, GenProg& p) {
    NetDims d{};
    d.L = mlp->n_layers; d.kin = mlp->dims[0]; d.obs_mode = mlp->obs_mode; d.n_out = mlp->dims[mlp->n_layers]; d.act = mlp->activation;
    for (int l = 0; l + 1 < mlp->n_layers; ++l) d.hid[l] = mlp->dims[l + 1];
    p = make_prog(d, split, fb);
    p.obs_scale = mlp->obs_log2_scale;
}

struct GenWorkspace {
    int64_t himg[GN_MAXL], dlimg[GN_MAXL], scale, img, masks, total;
};
static GenWorkspace gen_workspace(const b2048_mlp_desc* mlp, int64_t chunk, int num_sms) {
    GenWorkspace w;
    memset(&w, 0, sizeof(w));
    const int L = mlp->n_layers;
    const int64_t tiles = (chunk + TC_M - 1) / TC_M;
    int64_t o = 0;
    for (int l = 0; l < L - 1; ++l) { w.himg[l] = o; o += tiles * (mlp->dims[l + 1] / 64) * GN_SLAB; }
    for (int l = 0; l < L; ++l) { w.dlimg[l] = o; o += tiles * (l == L - 1 ? 1 : mlp->dims[l + 1] / 64) * GN_SLAB; }
    w.scale = o; o += 1024;
    GenProg p;
    build_program(mlp, true, true, p);
    w.img = o; o += ((int64_t)p.img_bytes + 1023) / 1024 * 1024;
    w.masks = o; o += (int64_t)num_sms * GN_MASK_WORDS * (mlp->activation == B2048_ACTV_SIGMOID ? 32 : 2);
    w.total = o;
    return w;
}
int64_t gen_workspace_bytes(const b2048_mlp_desc* mlp, int64_t chunk) { return gen_workspace(mlp, chunk, 256).total + 2048; }

static int gen_attrs(b2048_handle* h) {
    if (!(h->attrs & ATTR_GEN)) {
        cudaError_t e = cudaSuccess;
        auto set = [&](const void* f) { if (e == cudaSuccess) e = cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, GS_TOTAL); };
        set((const void*)gen_mlp_kernel<B2048_ACTV_RELU, false, 0, false, false>);
        set((const void*)gen_mlp_kernel<B2048_ACTV_SIGMOID, false, 0, false, false>);
        set((const void*)gen_mlp_kernel<B2048_ACTV_RELU, true, 0, false, false>);
        set((const void*)gen_mlp_kernel<B2048_ACTV_SIGMOID, true, 0, false, false>);
        set((const void*)gen_mlp_kernel<B2048_ACTV_RELU, false, 1, false, false>);
        set((const void*)gen_mlp_kernel<B2048_ACTV_RELU, false, 1, true, false>);
        set((const void*)gen_mlp_kernel<B2048_ACTV_RELU, false, 1, true, true>);
        set((const void*)gen_mlp_ent_kernel<B2048_ACTV_RELU, 0, false, false>);
        set((const void*)gen_mlp_ent_kernel<B2048_ACTV_SIGMOID, 0, false, false>);
        set((const void*)gen_mlp_ent_kernel<B2048_ACTV_RELU, 1, true, true>);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(gen_mlp_kernel)");
        e = cudaFuncSetAttribute(gen_dw_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
        if (e != cudaSuccess) return check_cuda(e, "cudaFuncSetAttribute(gen_dw_kernel)");
        h->attrs |= ATTR_GEN;
    }
    return B2048_OK;
}

static int gen_prepare(const b2048_mlp_desc* mlp, const GenProg& p, uint8_t* img, cudaStream_t stream) {
    GenPrepArgs pa;
    pa.p = p;
    for (int l = 0; l < GN_MAXL; ++l) { pa.W[l] = l < mlp->n_layers ? mlp->W[l] : nullptr; pa.b[l] = l < mlp->n_layers ? mlp->b[l] : nullptr; }
    for (int l = 0; l <= GN_MAXL; ++l) pa.dims[l] = l <= mlp->n_layers ? mlp->dims[l] : 0;
    pa.img = img;
    gen_prepare_kernel<<<128, 256, 0, stream>>>(pa);
    return check_cuda(cudaGetLastError(), "gen_prepare_kernel launch");
}

static int ensure_gen_image(b2048_handle* h, size_t bytes) {
    if (h->gen_image && h->gen_image_bytes >= bytes) return B2048_OK;
    if (h->gen_image) { cudaDeviceSynchronize(); cudaFree(h->gen_image); h->gen_image = nullptr; h->gen_image_bytes = 0; }
    const size_t cap = (bytes + (1u << 20)) & ~(size_t)((1u << 20) - 1);
    cudaError_t e = cudaMalloc(&h->gen_image, cap);
    if (e != cudaSuccess) return check_cuda(e, "cudaMalloc(gen_image)");
    h->gen_image_bytes = cap;
    return B2048_OK;
}

static int gen_dbg_print(const b2048_handle* h, const GenArgs& a, cudaStream_t stream) {
    if (!a.dbg) return B2048_OK;
    long long hb[256];
    { int st = debug_clock_read(h, hb, 256, stream); if (st != B2048_OK) return st; }
    for (int lt = 0; lt < 4; ++lt) {
        const long long* d = hb + 64 * lt;
        const long long t0 = d[0];
        if (t0 == 0) continue;
        fprintf(stderr, "[gen_mlp clock] tile %d (cycles from the MMA lane's tile start): io: loop top %lld loads done %lld input written %lld head ready %lld "
                        "tile end %lld\n", lt, d[60] - t0, d[61] - t0, d[62] - t0, d[63] - t0, d[59] - t0);
        for (int G = 0; G < a.p.n_gemm; ++G)
            fprintf(stderr, "    GEMM %d (%s layer %d, N %d, %d fills): A ready %lld, all MMAs issued %lld (weight waits %lld) | epilogue: acc ready %lld done %lld\n",
                    G, a.p.gemm[G].bwd ? "bwd" : "fwd", a.p.gemm[G].layer, a.p.gemm[G].N, a.p.gemm[G].nf, d[1 + 3 * G] - t0, d[2 + 3 * G] - t0,
                    d[3 + 3 * G], a.p.gemm[G].head ? 0 : d[32 + 2 * G] - t0, a.p.gemm[G].head ? 0 : d[33 + 2 * G] - t0);
    }
    return B2048_OK;
}

static void gen_launch(const GenArgs& a, int grid, cudaStream_t stream) {
    const bool sig = a.p.act == B2048_ACTV_SIGMOID;
    const GenProg& p = a.p;
    // the network whose program is compiled in (SpecProg<1>): one-hot 272-256-128-64, ReLU
    const bool spec1 = !sig && !a.dbg && p.L == 4 && p.kin == 272 && p.obs_mode == B2048_OBS_ONEHOT && p.width[0] == 256 && p.width[1] == 128 &&
                       p.width[2] == 64 && (p.fb == 0 || p.split == 1);
    if (spec1) {
        if (p.fb) gen_mlp_kernel<B2048_ACTV_RELU, false, 1, true, true><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
        else if (p.split) gen_mlp_kernel<B2048_ACTV_RELU, false, 1, true, false><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
        else gen_mlp_kernel<B2048_ACTV_RELU, false, 1, false, false><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
    } else if (a.dbg) {
        if (sig) gen_mlp_kernel<B2048_ACTV_SIGMOID, true, 0, false, false><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
        else gen_mlp_kernel<B2048_ACTV_RELU, true, 0, false, false><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
    } else {
        if (sig) gen_mlp_kernel<B2048_ACTV_SIGMOID, false, 0, false, false><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
        else gen_mlp_kernel<B2048_ACTV_RELU, false, 0, false, false><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
    }
}

// update mode with the entropy bonus: the kernels of gen_launch's update-mode choices without the debug clocks
static void gen_launch_ent(const GenEntArgs& a, int grid, cudaStream_t stream) {
    const GenProg& p = a.g.p;
    const bool sig = p.act == B2048_ACTV_SIGMOID;
    const bool spec1 = !sig && p.L == 4 && p.kin == 272 && p.obs_mode == B2048_OBS_ONEHOT && p.width[0] == 256 && p.width[1] == 128 &&
                       p.width[2] == 64 && p.split == 1;
    if (spec1) gen_mlp_ent_kernel<B2048_ACTV_RELU, 1, true, true><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
    else if (sig) gen_mlp_ent_kernel<B2048_ACTV_SIGMOID, 0, false, false><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
    else gen_mlp_ent_kernel<B2048_ACTV_RELU, 0, false, false><<<grid, GN_THREADS, GS_TOTAL, stream>>>(a);
}

static void gen_fill_common(GenArgs& a, const b2048_mlp_desc* mlp, const GenProg& p) {
    memset(&a, 0, sizeof(a));
    a.p = p;
    for (int l = 0; l < mlp->n_layers; ++l) a.bias[l] = mlp->b[l];
}

// Forward-only launch behind b2048_mlp_forward (split != 0: float32 grade, precision 3 / auto; else one fp16 MMA per product,
// precision 1) and b2048_policy_step (precision 1: logits -> masked softmax -> sample / greedy).  B2048_ERR_UNSUPPORTED
// (silent) for shapes outside gen_supported().
int launch_forward_gen(b2048_handle* h, const b2048_mlp_desc* mlp, const uint64_t* board, const uint8_t* mask_flags, float* out,
                       uint8_t* action, float* probs, float* logits, int64_t n, uint64_t seed, uint64_t gid0, uint32_t t, int greedy,
                       int split, bool rebuild_image, cudaStream_t stream, const int32_t* slot_map, const int32_t* n_dev) {
    if (!gen_supported(h, mlp) || (n < 4096 && slot_map == nullptr)) return B2048_ERR_UNSUPPORTED;
    { int st = gen_attrs(h); if (st != B2048_OK) return st; }
    GenProg p;
    build_program(mlp, split != 0, false, p);
    // one image area per precision so that a policy image (single) and a value image (split) do not evict each other
    const size_t half = (size_t)2 << 20;
    { int st = ensure_gen_image(h, 2 * half); if (st != B2048_OK) return st; }
    if (p.img_bytes > half) return B2048_ERR_UNSUPPORTED;
    uint8_t* img = h->gen_image + (split ? half : 0);
    if (rebuild_image) { int st = gen_prepare(mlp, p, img, stream); if (st != B2048_OK) return st; }
    GenArgs a;
    gen_fill_common(a, mlp, p);
    a.img = img; a.board = board; a.n = n;
    a.out = out; a.action = action; a.probs = probs; a.logits = logits; a.mask_flags = mask_flags;
    a.keys = make_keys(seed); a.gid0 = gid0; a.t = t; a.greedy = greedy;
    a.slot_map = slot_map; a.n_dev = slot_map ? n_dev : nullptr;
    const int64_t tiles = (n + TC_M - 1) / TC_M;
    const int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
    a.dbg = debug_clock_begin(h, B2048_DBG_TC_CLOCKS, stream);
    gen_launch(a, grid, stream);
    const int st = check_cuda(cudaGetLastError(), "gen_mlp_kernel launch");
    return st != B2048_OK ? st : gen_dbg_print(h, a, stream);
}

// Same contract as the fp32 body of b2048_mlp_backward (grads accumulated; flat layout W_0, b_0, W_1, b_1, ...).
int launch_backward_gen(b2048_handle* h, const uint64_t* board, const uint8_t* mask_flags, const uint8_t* action, const float* coef,
                        const b2048_mlp_desc* mlp, float* grads, int64_t n, int head_mode, uint8_t* workspace, int64_t chunk,
                        cudaStream_t stream, const float* ent_coef, double* ent_sum) {
    { int st = gen_attrs(h); if (st != B2048_OK) return st; }
    const int L = mlp->n_layers;
    uint8_t* ws = reinterpret_cast<uint8_t*>(((uintptr_t)workspace + 1023) & ~(uintptr_t)1023);
    const GenWorkspace w = gen_workspace(mlp, chunk, 256);
    GenProg p;
    build_program(mlp, true, true, p);
    { int st = gen_prepare(mlp, p, ws + w.img, stream); if (st != B2048_OK) return st; }
    float* scale = reinterpret_cast<float*>(ws + w.scale);
    { int st = launch_loss_scale(h, coef, n, scale, stream, ent_coef); if (st != B2048_OK) return st; }
    float *gW[B2048_MAX_LAYERS], *gb[B2048_MAX_LAYERS];
    carve_grads(mlp, grads, gW, gb);
    for (int64_t c0 = 0; c0 < n; c0 += chunk) {
        const int64_t cn = (n - c0) < chunk ? (n - c0) : chunk;
        const int64_t tiles = (cn + TC_M - 1) / TC_M;
        const int grid = (int)(tiles < h->num_sms ? tiles : h->num_sms);
        GenArgs a;
        gen_fill_common(a, mlp, p);
        a.img = ws + w.img; a.board = board + c0; a.n = cn;
        a.mask_flags = mask_flags ? mask_flags + c0 : nullptr;
        a.act_in = action ? action + c0 : nullptr;
        a.coef = coef + c0; a.scale = scale; a.head_mode = head_mode;
        for (int l = 0; l < L - 1; ++l) a.himg[l] = ws + w.himg[l];
        for (int l = 0; l < L; ++l) a.dlimg[l] = ws + w.dlimg[l];
        a.gb_head = gb[L - 1];
        if (mlp->activation == B2048_ACTV_SIGMOID) a.dsig_scratch = reinterpret_cast<uint4*>(ws + w.masks);
        else a.mask_scratch = reinterpret_cast<uint16_t*>(ws + w.masks);
        if (ent_coef) {                              // the entropy kernels carry no phase clocks
            GenEntArgs ea;
            ea.g = a; ea.e.ent_coef = ent_coef + c0; ea.e.ent_sum = ent_sum;
            gen_launch_ent(ea, grid, stream);
        } else {
            if (c0 == 0) a.dbg = debug_clock_begin(h, B2048_DBG_TC_CLOCKS, stream);
            gen_launch(a, grid, stream);
        }
        int st = check_cuda(cudaGetLastError(), "gen_mlp_kernel launch");
        if (st != B2048_OK || (st = gen_dbg_print(h, a, stream)) != B2048_OK) return st;
        for (int l = 0; l < L; ++l) {
            GenDwArgs d;
            memset(&d, 0, sizeof(d));
            const int K = mlp->dims[l];
            d.aimg = l == 0 ? nullptr : ws + w.himg[l - 1];
            d.board = board + c0; d.obs_mode = mlp->obs_mode; d.obs_scale = mlp->obs_log2_scale;
            d.bimg = ws + w.dlimg[l];
            d.a_slabs = (K + 63) / 64;
            d.b_slabs = l == L - 1 ? 1 : mlp->dims[l + 1] / 64;
            d.N = p.width[l];
            d.K_real = K; d.N_real = mlp->dims[l + 1];
            d.gW = gW[l]; d.gb = l == L - 1 ? nullptr : gb[l];
            d.inv_scale = scale + 1;
            d.n_tiles = tiles; d.n = cn;
            d.mtiles = (K + 127) / 128;
            int ksplit = h->num_sms / d.mtiles;
            if (ksplit < 1) ksplit = 1;
            if ((int64_t)ksplit > tiles) ksplit = (int)tiles;
            d.ksplit = ksplit;
            const int stage_bytes = (2 + d.b_slabs) * GN_SLAB;
            int stages = (227 * 1024 - 256) / stage_bytes;
            d.stages = stages > 4 ? 4 : stages;
            d.tmem_cols = d.N <= 32 ? 32u : (d.N <= 64 ? 64u : (d.N <= 128 ? 128u : 256u));
            const size_t smem = (size_t)d.stages * stage_bytes + 256;
            gen_dw_kernel<<<d.mtiles * d.ksplit, GD_THREADS, smem, stream>>>(d);
            st = check_cuda(cudaGetLastError(), "gen_dw_kernel launch");
            if (st != B2048_OK) return st;
        }
    }
    return B2048_OK;
}

}  // namespace b2
