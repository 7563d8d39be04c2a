// b2048_device.cuh — packed-board primitives shared by every kernel.
//
// A board is sixteen 4-bit exponents in a uint64 (cell (r,c) in nibble 4r+c), handled as two
// 32-bit words because the SM's integer datapath is 32 bits wide: lo = rows 0,1; hi = rows 2,3.
//
// Everything here is `B2_HD` (host+device) on purpose: tests/host_check compiles this header with
// g++ and checks the bit tricks against the CPU oracle on millions of boards without a GPU.  The
// product only ever calls them from kernels.
//
// Reference semantics restated (paths relative to the reference repo):
//   move        Game2048._move / _board_move_left / _row_move_left   src/game2048.py:120-165
//   legal mask  Game2048.get_action_mask                             src/game2048.py:95-99, :189-237
//   done        Game2048._is_done                                    src/game2048.py:172-187
//   spawn       Game2048._spawn                                      src/game2048.py:108-118
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define B2_HD __host__ __device__ __forceinline__
#else
#define B2_HD static inline
#endif

namespace b2 {

struct Board {
    uint32_t lo, hi;
};

B2_HD Board make_board(uint64_t b) { return Board{(uint32_t)b, (uint32_t)(b >> 32)}; }
B2_HD uint64_t to_u64(Board b) { return (uint64_t)b.lo | ((uint64_t)b.hi << 32); }

// ---------------------------------------------------------------- portable intrinsics
B2_HD uint32_t prmt(uint32_t x, uint32_t y, uint32_t s) {
#if defined(__CUDA_ARCH__)
    uint32_t r;  // raw PRMT: selectors here never set the sign-replicate bit, so no "& 0x7777" is needed
    asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(x), "r"(y), "r"(s));
    return r;
#else
    uint64_t v = (uint64_t)x | ((uint64_t)y << 32);
    uint32_t r = 0;
    for (int i = 0; i < 4; ++i) r |= (uint32_t)((v >> (8 * ((s >> (4 * i)) & 7))) & 0xFF) << (8 * i);
    return r;
#endif
}
B2_HD int popc(uint32_t x) {
#if defined(__CUDA_ARCH__)
    return __popc(x);
#else
    return __builtin_popcount(x);
#endif
}
B2_HD uint32_t mulhi(uint32_t a, uint32_t b) {
#if defined(__CUDA_ARCH__)
    return __umulhi(a, b);
#else
    return (uint32_t)(((uint64_t)a * b) >> 32);
#endif
}
B2_HD int ffs0(uint32_t x) {  // index of lowest set bit, x != 0
#if defined(__CUDA_ARCH__)
    return __ffs((int)x) - 1;
#else
    return __builtin_ctz(x);
#endif
}
// low 32 bits of ((hi:lo) >> s), 0 <= s < 32
B2_HD uint32_t funnel_r(uint32_t lo, uint32_t hi, uint32_t s) {
#if defined(__CUDA_ARCH__)
    return __funnelshift_r(lo, hi, s);
#else
    return s ? (lo >> s) | (hi << (32 - s)) : lo;
#endif
}

// x >> K for a compile-time K, issued on the FMA pipe (IMAD.HI by 2^(32-K)) instead of the integer ALU pipe:
// the step kernel is bound by the ALU pipe (LOP3 / SHF / IADD3 at 16 lanes per clock per scheduler), the FMA pipe
// is nearly idle, and ptxas keeps mul.hi with an immediate as IMAD.HI.U32.
template <int K>
B2_HD uint32_t shr_fma(uint32_t x) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("mul.hi.u32 %0, %1, %2;" : "=r"(r) : "r"(x), "n"(1u << (32 - K)));
    return r;
#else
    return x >> K;
#endif
}

// (on1 & mask) | (on0 & ~mask) in one LOP3
B2_HD uint32_t bitsel(uint32_t mask, uint32_t on1, uint32_t on0) {
#if defined(__CUDA_ARCH__)
    uint32_t r;
    asm("lop3.b32 %0, %1, %2, %3, 0xE4;" : "=r"(r) : "r"(on1), "r"(on0), "r"(mask));
    return r;
#else
    return (on1 & mask) | (on0 & ~mask);
#endif
}

// bit 3 of every nibble set iff that nibble is non-zero (exact, no cross-nibble carry)
B2_HD uint32_t nz8(uint32_t x) { return (((x & 0x77777777u) + 0x77777777u) | x) & 0x88888888u; }

// ---------------------------------------------------------------- Philox4x32-10
struct Rand4 {
    uint32_t w0, w1, w2, w3;
};

B2_HD Rand4 philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint32_t h0 = mulhi(M0, c0), l0 = M0 * c0;
        uint32_t h1 = mulhi(M1, c2), l1 = M1 * c2;
        c0 = h1 ^ c1 ^ k0;
        c1 = l1;
        c2 = h0 ^ c3 ^ k1;
        c3 = l0;
        k0 += W0;
        k1 += W1;
    }
    return Rand4{c0, c1, c2, c3};
}

// Round keys k_r = key + r * (W0, W1), computed once on the host and passed by value in the kernel
// arguments so the per-board Philox block spends no instructions on the key schedule.
struct PhiloxKeys {
    uint32_t k0[10], k1[10];
};
B2_HD PhiloxKeys make_keys(uint64_t seed) {
    PhiloxKeys k;
    uint32_t a = (uint32_t)seed, b = (uint32_t)(seed >> 32);
    for (int r = 0; r < 10; ++r) { k.k0[r] = a; k.k1[r] = b; a += 0x9E3779B9u; b += 0xBB67AE85u; }
    return k;
}
B2_HD Rand4 philox_keyed(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const PhiloxKeys& k) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        c0 = (uint32_t)(p1 >> 32) ^ c1 ^ k.k0[r];
        c1 = (uint32_t)p1;
        c2 = (uint32_t)(p0 >> 32) ^ c3 ^ k.k1[r];
        c3 = (uint32_t)p0;
    }
    return Rand4{c0, c1, c2, c3};
}
B2_HD Rand4 stream_keyed(const PhiloxKeys& k, uint64_t gid, uint32_t t, uint32_t domain) {
    return philox_keyed((uint32_t)gid, (uint32_t)(gid >> 32), t, domain, k);
}

B2_HD Rand4 stream(uint64_t seed, uint64_t gid, uint32_t t, uint32_t domain) {
    return philox4x32_10((uint32_t)gid, (uint32_t)(gid >> 32), t, domain, (uint32_t)seed, (uint32_t)(seed >> 32));
}

// ---------------------------------------------------------------- canonicalisation
// Every move is reduced to "slide each 16-bit row toward nibble 0" by a conditional transpose
// (vertical moves) and a conditional mirror (right/down), both branch-free: the nibble-level parts
// use a data-dependent shift amount (0 = identity) and the byte-level parts a data-dependent PRMT
// selector, so lanes of a warp playing different actions never diverge.
//
//   a : 0 up (transpose), 1 right (mirror), 2 down (transpose+mirror), 3 left (identity)
struct Xform {
    uint32_t st;      // 12 if vertical else 0   (2x2 in-block transpose shift)
    uint32_t sm;      // 4 if mirror else 0      (nibble swap shift)
    uint32_t f_lo, f_hi, i_lo, i_hi;  // PRMT selectors: forward / inverse byte permutation
};

B2_HD Xform xform_for(uint32_t a) {
    // per-action selectors packed 16 bits each (action a in bits [16a, 16a+16))
    const uint64_t F_LO = 0x3210260423016240ull, F_HI = 0x7654371567457351ull;
    const uint64_t I_LO = 0x3210735123016240ull, I_HI = 0x7654624067457351ull;
    uint32_t sh = 16u * a;
    Xform x;
    x.st = (a & 1u) ? 0u : 12u;
    x.sm = ((a ^ (a >> 1)) & 1u) ? 4u : 0u;
    x.f_lo = (uint32_t)(F_LO >> sh);
    x.f_hi = (uint32_t)(F_HI >> sh);
    x.i_lo = (uint32_t)(I_LO >> sh);
    x.i_hi = (uint32_t)(I_HI >> sh);
    return x;
}

B2_HD uint32_t blk_transpose(uint32_t x, uint32_t s) {  // s in {0,12}
    return bitsel(0x0F0F0000u, x << s, bitsel(0x0000F0F0u, x >> s, x));  // the three masks partition the word
}
B2_HD uint32_t nib_swap(uint32_t x, uint32_t s) {  // s in {0,4}
    return bitsel(0xF0F0F0F0u, x << s, x >> s);
}
// The same two transforms without a data-dependent shift, for the ALU-bound fast step: the shifts become IMADs on
// the FMA pipe and the choice between transform and identity moves into per-action masks / multipliers.
//   blk_transpose_m(x, tm) == blk_transpose(x, s) for tm = 0x0F0F0000 (s = 12) or 0 (s = 0)
//   nib_swap_m(x, nl, nr)  == nib_swap(x, s)      for (nl, nr) = (16, 1) (s = 4) or (1, 16) (s = 0);
// with s = 0, (x * 16) >> 4 drops only the top nibble, which the 0x0F0F0F0F half of the select does not keep.
B2_HD uint32_t blk_transpose_m(uint32_t x, uint32_t tm) {
    return bitsel(tm, x * 4096u, bitsel(shr_fma<12>(tm), shr_fma<12>(x), x));
}
B2_HD uint32_t nib_swap_m(uint32_t x, uint32_t nl, uint32_t nr) {
    return bitsel(0xF0F0F0F0u, x * nl, shr_fma<4>(x * nr));
}

B2_HD Board canon_fwd(Board b, const Xform& x) {
    uint32_t lo = nib_swap(blk_transpose(b.lo, x.st), x.sm);
    uint32_t hi = nib_swap(blk_transpose(b.hi, x.st), x.sm);
    return Board{prmt(lo, hi, x.f_lo), prmt(lo, hi, x.f_hi)};
}
B2_HD Board canon_inv(Board b, const Xform& x) {
    uint32_t lo = prmt(b.lo, b.hi, x.i_lo), hi = prmt(b.lo, b.hi, x.i_hi);
    return Board{blk_transpose(nib_swap(lo, x.sm), x.st), blk_transpose(nib_swap(hi, x.sm), x.st)};
}

// ---------------------------------------------------------------- row tables
// lut_left[row]  : row after sliding toward nibble 0
// lut_merge[row] : nibble 0 = exponent of the first merged tile, nibble 1 = second; 0 none,
//                  1 = the out-of-domain exponent 16 (15+15)
// Single source of truth for one row (used by the table-building kernel and by host_check).
B2_HD void row_move_left(uint32_t row, uint32_t& out, uint32_t& merge) {
    uint32_t cells[4];
    int n = 0;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
        uint32_t e = (row >> (4 * c)) & 0xFu;
        if (e) cells[n++] = e;
    }
    out = 0;
    merge = 0;
    int i = 0, w = 0, nm = 0;
    while (i < n) {
        if (i + 1 < n && cells[i] == cells[i + 1]) {
            uint32_t e = cells[i] + 1;
            out |= (e > 15u ? 15u : e) << (4 * w);
            merge |= (e > 15u ? 1u : e) << (4 * nm);
            ++nm;
            i += 2;
        } else {
            out |= cells[i] << (4 * w);
            i += 1;
        }
        ++w;
    }
}

struct MoveResult {
    Board board;     // board after the move (before any spawn)
    uint32_t merge;  // eight nibbles: two per canonical row (see lut_merge)
};

// Tables are passed as generic pointers: shared-memory staged copy in the large-batch kernels,
// the global (L2-resident) copy in the small-batch / preview kernels.
template <typename LutL, typename LutM>
B2_HD MoveResult move_board(Board b, uint32_t a, LutL lut_left, LutM lut_merge) {
    Xform x = xform_for(a);
    Board c = canon_fwd(b, x);
    uint32_t i0 = c.lo & 0xFFFFu, i1 = c.lo >> 16, i2 = c.hi & 0xFFFFu, i3 = c.hi >> 16;
    uint32_t r0 = lut_left[i0], r1 = lut_left[i1], r2 = lut_left[i2], r3 = lut_left[i3];
    uint32_t m0 = lut_merge[i0], m1 = lut_merge[i1], m2 = lut_merge[i2], m3 = lut_merge[i3];
    Board moved{r0 | (r1 << 16), r2 | (r3 << 16)};
    MoveResult res;
    res.board = canon_inv(moved, x);
    res.merge = m0 | (m1 << 8) | (m2 << 16) | (m3 << 24);
    return res;
}

// ---------------------------------------------------------------- merge statistics
struct MergeStats {
    uint32_t n;         // number of merges                 (len(merged), env.py:234)
    uint32_t sum_log2;  // sum of merged exponents          (env.py:218-220)
    uint32_t sum;       // sum of merged tile values        (game2048.py:167-170)
    uint32_t max_exp;   // largest merged exponent, 0 none  (env.py:239)
    bool overflow;      // a 15+15 merge happened
};

B2_HD MergeStats merge_stats(uint32_t m, bool want_sum, bool want_max) {
    MergeStats s;
    uint32_t nzb = nz8(m);
    s.n = (uint32_t)popc(nzb);
    // sentinel nibble == 1 means exponent 16
    uint32_t is1 = nzb & ~nz8(m ^ 0x11111111u);  // nibble == 1  <=> m^1 == 0 and (trivially) m != 0
    s.overflow = is1 != 0u;
    uint32_t pairs = (m & 0x0F0F0F0Fu) + ((m >> 4) & 0x0F0F0F0Fu);
    pairs = (pairs & 0x00FF00FFu) + ((pairs >> 8) & 0x00FF00FFu);
    s.sum_log2 = (pairs + (pairs >> 16)) & 0xFFFFu;
    s.sum = 0;
    s.max_exp = 0;
    if (s.overflow) s.sum_log2 += 15u * (uint32_t)popc(is1);
    if (want_sum || want_max) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            uint32_t e = (m >> (4 * k)) & 0xFu;
            e = (e == 1u) ? 16u : e;
            if (want_sum) s.sum += e ? (1u << e) : 0u;
            if (want_max) s.max_exp = e > s.max_exp ? e : s.max_exp;
        }
    }
    return s;
}

// ---------------------------------------------------------------- legal mask / done
// bit a set iff action a changes the board.  Slides: a line can slide iff somewhere an empty cell
// has a non-empty cell on its far side; adjacent (empty, tile) pairs are sufficient to test.
// Merges: adjacent equal non-empty cells.  All sixteen non-zero bits are packed into ONE word
// (rows 0,1 at bit 3 of each nibble, rows 2,3 shifted to bit 2), so each test is one LOP3.
B2_HD uint32_t legal_mask(Board b) {
    uint32_t n_lo = nz8(b.lo), n_hi = nz8(b.hi);
    uint32_t N = n_lo | (n_hi >> 1);  // rows 0,1: bits 4i+3 ; rows 2,3: bits 4i+2
    // horizontal neighbours: cell i+1 aligned onto cell i (valid for columns 0..2)
    const uint32_t MH = 0x0CCC0CCCu;
    uint32_t Nr = N >> 4;
    uint32_t e_lo = b.lo ^ (b.lo >> 4), e_hi = b.hi ^ (b.hi >> 4);
    uint32_t EH = nz8(e_lo) | (nz8(e_hi) >> 1);
    uint32_t hmerge = ~EH & N & MH;
    uint32_t left = (~N & Nr & MH) | hmerge;   // empty at i, tile at i+1  -> slides toward col 0
    uint32_t right = (N & ~Nr & MH) | hmerge;  // tile at i, empty at i+1  -> slides toward col 3
    // vertical neighbours: cell (r+1,c) aligned onto (r,c) (valid for rows 0..2)
    // row0 bits 4c+3 (c<4), row1 bits 16+4c+3, row2 bits 4c+2, row3 bits 16+4c+2
    const uint32_t MV = 0x8888CCCCu;  // rows 0,1,2
    uint32_t Nd = ((N >> 16) & 0x0000CCCCu) | ((N << 17) & 0x88880000u);
    uint32_t v_lo = b.lo ^ funnel_r(b.lo, b.hi, 16), v_hi = b.hi ^ (b.hi >> 16);
    uint32_t EV = nz8(v_lo) | (nz8(v_hi) >> 1);
    uint32_t vmerge = ~EV & N & MV;
    uint32_t up = (~N & Nd & MV) | vmerge;    // empty above a tile -> slides toward row 0
    uint32_t down = (N & ~Nd & MV) | vmerge;  // tile above an empty -> slides toward row 3
    return (up ? 1u : 0u) | (right ? 2u : 0u) | (down ? 4u : 0u) | (left ? 8u : 0u);
}

B2_HD int count_empty(Board b) { return 16 - popc(nz8(b.lo)) - popc(nz8(b.hi)); }

// ---------------------------------------------------------------- spawn
// Places exponent `val` in the k-th empty cell in row-major order; k < number of empties.
B2_HD Board place_kth_empty(Board b, uint32_t k, uint32_t val) {
    uint32_t z_lo = ~nz8(b.lo) & 0x88888888u, z_hi = ~nz8(b.hi) & 0x88888888u;
    uint32_t c_lo = (uint32_t)popc(z_lo);
    bool in_hi = k >= c_lo;
    uint32_t z = in_hi ? z_hi : z_lo;
    k = in_hi ? k - c_lo : k;
    uint32_t pos = 0;
    uint32_t c = (uint32_t)popc(z & 0xFFFFu);
    if (k >= c) { k -= c; z >>= 16; pos += 4; }
    c = (uint32_t)popc(z & 0xFFu);
    if (k >= c) { k -= c; z >>= 8; pos += 2; }
    c = (z >> 3) & 1u;
    if (k >= c) pos += 1;
    uint32_t v = val << (4 * pos);
    if (in_hi) b.hi |= v; else b.lo |= v;
    return b;
}

// Game2048._spawn with the replayable draws (see include/b2048.h)
B2_HD Board spawn(Board b, uint32_t wp, uint32_t wv) {
    int n = count_empty(b);
    if (n == 0) return b;
    uint32_t k = mulhi(wp, (uint32_t)n);
    uint32_t val = wv >= 0xE6666667u ? 2u : 1u;
    return place_kth_empty(b, k, val);
}

B2_HD Board reset_board(uint64_t seed, uint64_t gid, uint32_t t) {
    Rand4 r = stream(seed, gid, t, 1u /* B2048_DOM_RESET */);
    Board b{0u, 0u};
    b = spawn(b, r.w0, r.w1);
    b = spawn(b, r.w2, r.w3);
    return b;
}

// first legal action in the order prio (nibble k = k-th choice), 0 if the mask is empty
// (tools/simple_action_gen.py:16-33)
B2_HD uint32_t pick_priority(uint32_t mask, uint32_t prio) {
    uint32_t a = 0u;
#pragma unroll
    for (int k = 3; k >= 0; --k) {
        uint32_t c = (prio >> (4 * k)) & 3u;
        a = ((mask >> c) & 1u) ? c : a;
    }
    return a;
}

// j-th (0-based) legal action of a 4-bit mask, 0 if the mask is empty
B2_HD uint32_t pick_legal(uint32_t mask, uint32_t w) {
    uint32_t n = (uint32_t)popc(mask & 0xFu);
    uint32_t j = mulhi(w, n);
    uint32_t m = mask & 0xFu;
    if (j >= 1) m &= m - 1;
    if (j >= 2) m &= m - 1;
    if (j >= 3) m &= m - 1;
    return m ? (uint32_t)ffs0(m) : 0u;
}

}  // namespace b2
