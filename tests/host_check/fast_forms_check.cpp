// Checks the closed forms of the fast step body (csrc/b2048_step_fast.cuh) against the generic primitives they replace
// (csrc/b2048_device.cuh), compiled with g++.  Each function returns the number of mismatches.
#include "../../rl-2048-with-reinforce-and-actor-critic_b200/csrc/b2048_step_fast.cuh"

static uint64_t splitmix(uint64_t& s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

static int64_t start_mismatch(const b2::Rand4& w) {
    const b2::Board ref = b2::spawn(b2::spawn(b2::Board{0u, 0u}, w.w0, w.w1), w.w2, w.w3);
    uint32_t mask = 0xFFu;
    const b2::Board got = b2::start_board(w, mask);
    return (got.lo != ref.lo || got.hi != ref.hi || mask != b2::legal_mask(ref)) ? 1 : 0;
}

extern "C" {

// start_board (board and legal mask) against the two spawns of reset_board and legal_mask: every (c1, k2, v1, v2),
// each at both ends of its range of words, then reset_board itself for boards gid0 .. gid0 + n - 1
int64_t hc_start_board_mismatches(int64_t n, uint64_t seed, uint64_t gid0, uint32_t t) {
    int64_t bad = 0;
    for (uint32_t c1 = 0; c1 < 16; ++c1)
        for (uint32_t k2 = 0; k2 < 15; ++k2) {
            const uint32_t w0[2] = {c1 << 28, (c1 << 28) | 0x0FFFFFFFu};
            // smallest / largest w with mulhi(w, 15) == k2
            const uint32_t w2[2] = {(uint32_t)(((uint64_t)k2 << 32) / 15 + (((uint64_t)k2 << 32) % 15 ? 1 : 0)),
                                    (uint32_t)((((uint64_t)(k2 + 1) << 32) + 14) / 15 - 1)};
            const uint32_t wv[4] = {0u, 0xE6666666u, 0xE6666667u, 0xFFFFFFFFu};   // value 2, 2, 4, 4
            for (int a = 0; a < 2; ++a)
                for (int b = 0; b < 2; ++b)
                    for (int u = 0; u < 4; ++u)
                        for (int v = 0; v < 4; ++v) bad += start_mismatch(b2::Rand4{w0[a], wv[u], w2[b], wv[v]});
        }
    const b2::PhiloxKeys keys = b2::make_keys(seed);
    for (int64_t i = 0; i < n; ++i) {
        const uint64_t gid = gid0 + (uint64_t)i;
        const b2::Board ref = b2::reset_board(seed, gid, t);
        uint32_t mask = 0xFFu;
        const b2::Board got = b2::start_board(b2::stream_keyed(keys, gid, t, B2048_DOM_RESET), mask);
        bad += (got.lo != ref.lo || got.hi != ref.hi || mask != b2::legal_mask(ref)) ? 1 : 0;
    }
    return bad;
}

// blk_transpose_m / nib_swap_m with the per-action SelEntry constants against blk_transpose / nib_swap with the
// Xform shifts, word by word and as the whole forward / inverse canonicalisation, for all 4 actions on n random boards
int64_t hc_canon_m_mismatches(int64_t n, uint64_t seed) {
    int64_t bad = 0;
    uint64_t s = seed;
    for (uint32_t a = 0; a < 4; ++a) {
        const b2::Xform x = b2::xform_for(a);
        b2::SelEntry e;
        b2::small_table_entry_sel(a, e);
        for (int64_t i = 0; i < n; ++i) {
            const b2::Board b = b2::make_board(splitmix(s));
            const uint32_t words[2] = {b.lo, b.hi};
            for (uint32_t w : words) {
                bad += b2::blk_transpose_m(w, e.tm) != b2::blk_transpose(w, x.st);
                bad += b2::nib_swap_m(w, e.nl, e.nr) != b2::nib_swap(w, x.sm);
            }
            const uint32_t clo = b2::nib_swap_m(b2::blk_transpose_m(b.lo, e.tm), e.nl, e.nr);
            const uint32_t chi = b2::nib_swap_m(b2::blk_transpose_m(b.hi, e.tm), e.nl, e.nr);
            const b2::Board f = b2::canon_fwd(b, x);
            bad += (b2::prmt(clo, chi, e.f_lo) != f.lo || b2::prmt(clo, chi, e.f_hi) != f.hi) ? 1 : 0;
            const uint32_t plo = b2::prmt(b.lo, b.hi, e.i_lo), phi = b2::prmt(b.lo, b.hi, e.i_hi);
            const b2::Board v = b2::canon_inv(b, x);
            bad += (b2::blk_transpose_m(b2::nib_swap_m(plo, e.nl, e.nr), e.tm) != v.lo ||
                    b2::blk_transpose_m(b2::nib_swap_m(phi, e.nl, e.nr), e.tm) != v.hi) ? 1 : 0;
        }
    }
    return bad;
}

}  // extern "C"
