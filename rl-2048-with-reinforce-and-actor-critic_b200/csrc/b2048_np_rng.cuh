// b2048_np_rng.cuh — NumPy's default_rng streams (PCG64 seeded through SeedSequence), one per board.
//
// The reference seeds every episode twice (runner.py:244-261): np.random.default_rng(env_seed) draws the spawns
// (Game2048._spawn, game2048.py:102-118: rng.integers(n_empty), then rng.random() >= 0.9 for a 4) and
// np.random.default_rng(policy_seed) draws the actions (rng.choice(4, p=probs), reinforce_agent.py:187).  This header
// restates exactly the NumPy arithmetic those calls run, so a batch of boards can play the reference's own seeded
// episodes on the device:
//   seed     SeedSequence(seed).generate_state(4, uint64) -> pcg64_set_seed (numpy/random/bit_generator.pyx, pcg64.c)
//   next64   pcg64_random_r: one 128-bit LCG step, then the XSL-RR output of the new state
//   next32   pcg64_next32: the high half of a 64-bit output is buffered in (has_uint32, uinteger)
//   random   (next64 >> 11) * 2^-53 (does not touch the buffer)
//   bounded  Generator.integers(n) for int64: nothing drawn for n == 1, else Lemire's method on next32
//   choice4  Generator.choice(4, p): float64 cumsum, divided by its last element, searchsorted(u, 'right')
// Host + device: tests/host_check compiles it with g++ and compares it with the installed NumPy.  No inline PTX: the
// 128-bit product is built from 64-bit halves (__umul64hi on the device).
#pragma once
#include "../../include/b2048.h"
#include "b2048_device.cuh"

namespace b2 {
namespace np {

constexpr uint64_t kMulHi = 0x2360ed051fc65da4ull;   // PCG_DEFAULT_MULTIPLIER_128
constexpr uint64_t kMulLo = 0x4385df649fccf645ull;

B2_HD uint64_t umulhi64(uint64_t a, uint64_t b) {
#if defined(__CUDA_ARCH__)
    return __umul64hi(a, b);
#else
    return (uint64_t)(((unsigned __int128)a * b) >> 64);
#endif
}

// state = state * MULT + inc  (mod 2^128)
B2_HD void step(b2048_np_rng& r) {
    const uint64_t lo = r.state_lo * kMulLo;
    const uint64_t hi = umulhi64(r.state_lo, kMulLo) + r.state_lo * kMulHi + r.state_hi * kMulLo;
    const uint64_t nlo = lo + r.inc_lo;
    r.state_hi = hi + r.inc_hi + (nlo < lo ? 1u : 0u);
    r.state_lo = nlo;
}

B2_HD uint64_t next64(b2048_np_rng& r) {
    step(r);
    const uint64_t x = r.state_hi ^ r.state_lo;
    const unsigned rot = (unsigned)(r.state_hi >> 58);
    return (x >> rot) | (x << ((64u - rot) & 63u));
}

B2_HD uint32_t next32(b2048_np_rng& r) {
    if (r.has_uint32) {
        r.has_uint32 = 0u;
        return r.uinteger;
    }
    const uint64_t x = next64(r);
    r.has_uint32 = 1u;
    r.uinteger = (uint32_t)(x >> 32);
    return (uint32_t)x;
}

B2_HD double next_double(b2048_np_rng& r) { return (double)(next64(r) >> 11) * (1.0 / 9007199254740992.0); }

// Generator.integers(n), 1 <= n < 2^32 (random_bounded_uint64_fill -> buffered_bounded_lemire_uint32 with rng = n - 1)
B2_HD uint32_t bounded(b2048_np_rng& r, uint32_t n) {
    if (n <= 1u) return 0u;
    uint64_t m = (uint64_t)next32(r) * n;
    uint32_t leftover = (uint32_t)m;
    if (leftover < n) {
        const uint32_t threshold = (0xFFFFFFFFu - (n - 1u)) % n;
        while (leftover < threshold) {
            m = (uint64_t)next32(r) * n;
            leftover = (uint32_t)m;
        }
    }
    return (uint32_t)(m >> 32);
}

// Game2048._spawn's two draws on a board with n_empty empty cells, encoded like spawn_replay:
// bits 0-3 = k (the k-th empty cell in row-major order), bit 4 = the tile is a 4.  Nothing is drawn without an empty cell.
B2_HD uint32_t spawn_draw(b2048_np_rng& r, uint32_t n_empty) {
    if (n_empty == 0u) return 0u;
    const uint32_t k = bounded(r, n_empty);
    const uint32_t four = next_double(r) >= 0.9 ? 1u : 0u;
    return k | (four << 4);
}

// Game2048._spawn on a board (the caller knows it has an empty cell when the move changed it)
B2_HD Board spawn(b2048_np_rng& r, Board b) {
    const uint32_t d = spawn_draw(r, (uint32_t)count_empty(b));
    return place_kth_empty(b, d & 0xFu, (d & 0x10u) ? 2u : 1u);
}

// Game2048.reset's board: two spawns on the empty board (16, then 15 empty cells)
B2_HD Board reset_board(b2048_np_rng& r) {
    Board b = spawn(r, Board{0u, 0u});
    return spawn(r, b);
}

// rng.choice(4, p=probs) with float32 probabilities
B2_HD uint32_t choice4(b2048_np_rng& r, float p0, float p1, float p2, float p3) {
    const double c0 = (double)p0, c1 = c0 + (double)p1, c2 = c1 + (double)p2, c3 = c2 + (double)p3;
    const double u = next_double(r);
    return (c0 / c3 <= u ? 1u : 0u) + (c1 / c3 <= u ? 1u : 0u) + (c2 / c3 <= u ? 1u : 0u) + (c3 / c3 <= u ? 1u : 0u);
}

// SeedSequence(seed) with its default pool of four 32-bit words (numpy/random/bit_generator.pyx)
B2_HD uint32_t hashmix(uint32_t v, uint32_t& hc) {
    v ^= hc;
    hc *= 0x931e8875u;   // MULT_A
    v *= hc;
    return v ^ (v >> 16);
}

B2_HD uint32_t mix(uint32_t x, uint32_t y) {
    uint32_t r = 0xca01f9ddu * x - 0x4973f715u * y;   // MIX_MULT_L, MIX_MULT_R
    return r ^ (r >> 16);
}

// default_rng(seed) for an integer seed in [0, 2^64): the entropy is the seed's 32-bit words, least significant first
B2_HD b2048_np_rng seed(uint64_t s) {
    const uint32_t ent[2] = {(uint32_t)s, (uint32_t)(s >> 32)};
    const int n_ent = (s >> 32) ? 2 : 1;
    uint32_t pool[4];
    uint32_t hc = 0x43b0d7e5u;   // INIT_A
    for (int i = 0; i < 4; ++i) pool[i] = hashmix(i < n_ent ? ent[i] : 0u, hc);
    for (int src = 0; src < 4; ++src)
        for (int dst = 0; dst < 4; ++dst)
            if (src != dst) pool[dst] = mix(pool[dst], hashmix(pool[src], hc));
    // generate_state(4, np.uint64): eight 32-bit words, paired little-endian into four uint64
    uint32_t w[8];
    uint32_t hb = 0x8b51f9ddu;   // INIT_B
    for (int i = 0; i < 8; ++i) {
        uint32_t v = pool[i & 3] ^ hb;
        hb *= 0x58f38dedu;   // MULT_B
        v *= hb;
        w[i] = v ^ (v >> 16);
    }
    uint64_t v64[4];
    for (int i = 0; i < 4; ++i) v64[i] = (uint64_t)w[2 * i] | ((uint64_t)w[2 * i + 1] << 32);
    // pcg64_set_seed -> pcg_setseq_128_srandom_r(initstate = v0:v1, initseq = v2:v3)
    b2048_np_rng r;
    r.inc_hi = (v64[2] << 1) | (v64[3] >> 63);
    r.inc_lo = (v64[3] << 1) | 1u;
    r.state_hi = 0u;
    r.state_lo = 0u;
    step(r);
    const uint64_t lo = r.state_lo + v64[1];
    r.state_hi = r.state_hi + v64[0] + (lo < r.state_lo ? 1u : 0u);
    r.state_lo = lo;
    step(r);
    r.has_uint32 = 0u;
    r.uinteger = 0u;
    r.reserved = 0u;
    return r;
}

}  // namespace np
}  // namespace b2
