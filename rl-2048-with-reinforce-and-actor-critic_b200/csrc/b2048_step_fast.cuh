// b2048_step_fast.cuh — instruction-lean body of the fused env step for the action-mask-on configurations
// (every reward term of env.py:197-261 except the invalid-action penalty of mask-off envs; the new-max-tile bonus needs
// the tracked counters; no observation / float64 / replay outputs).
//
// Same semantics as step_one (b2048_step.cuh; reference src/game2048.py:40-70, src/env.py:197-302) —
// the two are checked against each other and against the CPU oracle by tests/host_check — but built
// to minimise issued instructions and the length of their dependent chains, which is what bounds the step kernel on
// sm_100 (profiles/; a shift issued as IMAD.HI on the FMA pipe instead of SHF measured slower, not faster):
//   * per-action transform constants come from a 4-entry table (two 128-bit loads), not bit arithmetic;
//   * merge statistics (score, sum of log2, count, max, overflow) come from a 256-entry table indexed by
//     each row's merge byte and are combined with two adds and two ors;
//   * the spawn cell is found with one multiply-prefix-sum per half and one nibble-lane compare, and the
//     isolated bit (G & -G) is turned into the tile with one multiply (no find-first-set, no shifts);
//   * the non-zero masks of the moved board are reused for the legal-move test of the new board;
//   * the canonicalisation has no data-dependent shift (blk_transpose_m / nib_swap_m: multiplies and per-action masks);
//   * auto-reset looks the two-tile start board and its legal mask up by the cells and values its Philox words pick
//     (start_board) instead of running the generic reset_board + legal_mask.
// Host+device like the other step headers.
#pragma once
#include "b2048_step.cuh"

namespace b2 {

// ---- small tables appended to the row tables (built once by build_small_tables) -----------------
struct SelEntry {            // per action (0 up, 1 right, 2 down, 3 left)
    uint32_t f_lo, f_hi, i_lo, i_hi;   // PRMT selectors forward / inverse
    uint32_t tm, nl, nr, pad;          // blk_transpose_m mask, nib_swap_m multipliers (b2048_device.cuh)
};
struct AggEntry {            // per merge byte (two 4-bit merged exponents; 0 none, 1 = exponent 16)
    uint32_t agg;            // bits 0-19 sum of merged tiles, 20-27 sum of exponents, 28-31 count
    uint32_t orm;            // OR of (1 << exponent)
};
#define B2048_SMALL_AGG_OFF 0
#define B2048_SMALL_SEL_OFF 2048
#define B2048_SMALL_ACT_OFF (2048 + 128)
#define B2048_SMALL_BYTES (2048 + 128 + 64)   // multiple of 16

B2_HD void small_table_entry_agg(uint32_t byte, AggEntry& e) {
    e.agg = 0; e.orm = 0;
    for (int k = 0; k < 2; ++k) {
        uint32_t m = (byte >> (4 * k)) & 0xFu;
        if (!m) continue;
        uint32_t ex = m == 1u ? 16u : m;
        e.agg += (1u << ex) + (ex << 20) + (1u << 28);
        e.orm |= 1u << ex;
    }
}
B2_HD void small_table_entry_sel(uint32_t a, SelEntry& s) {
    Xform x = xform_for(a);
    s.f_lo = x.f_lo & 0xFFFFu; s.f_hi = x.f_hi & 0xFFFFu; s.i_lo = x.i_lo & 0xFFFFu; s.i_hi = x.i_hi & 0xFFFFu;
    s.tm = x.st ? 0x0F0F0000u : 0u;
    s.nl = x.sm ? 16u : 1u;
    s.nr = x.sm ? 1u : 16u;
    s.pad = 0;
}
// T_act[mask * 4 + j] = j-th legal action of the 4-bit mask (0 when j is out of range)
B2_HD uint32_t small_table_entry_act(uint32_t mask, uint32_t j) {
    uint32_t m = mask;
    for (uint32_t q = 0; q < j; ++q) m &= m - 1;
    return m ? (uint32_t)ffs0(m) : 0u;
}

// ---- auto-reset by table lookup --------------------------------------------------------------------
// reset_board(seed, gid, t) spawns on the empty board from the words w of stream(seed, gid, t, B2048_DOM_RESET): the
// first tile goes to cell c1 = mulhi(w0, 16), the second to the k2-th (k2 = mulhi(w2, 15)) of the 15 cells left, that
// is cell c2 = k2 + (k2 >= c1); a tile is 4 (exponent 2) when its value word is >= 0xE6666667, else 2.  start_board
// looks the board and its legal mask up by (c1, k2, v1, v2) instead of two place_kth_empty and a legal_mask.  The
// tables sit in constant memory: only the lanes that reset read them, so the step kernels stage nothing more into
// shared memory for them.
struct StartTables {               // index (c1 * 16 + k2) * 4 + 2 * (v1 - 1) + (v2 - 1)
    Board board[1024];
    uint8_t mask[1024];
};
// legal mask of a board given cell by cell (exponent per cell, row-major): bit a set iff some tile has an empty or
// equal neighbour in direction a (0 up, 1 right, 2 down, 3 left).  Plain loops, so it can build the tables at compile time.
constexpr uint32_t cells_legal_mask(const uint8_t (&e)[16]) {
    const int dr[4] = {-1, 0, 1, 0}, dc[4] = {0, 1, 0, -1};
    uint32_t m = 0;
    for (int c = 0; c < 16; ++c)
        for (int a = 0; a < 4; ++a) {
            const int r2 = c / 4 + dr[a], c2 = c % 4 + dc[a];
            if (e[c] && r2 >= 0 && r2 < 4 && c2 >= 0 && c2 < 4 && (e[4 * r2 + c2] == 0 || e[4 * r2 + c2] == e[c])) m |= 1u << a;
        }
    return m;
}
constexpr StartTables make_start_tables() {
    StartTables s{};
    for (uint32_t c1 = 0; c1 < 16; ++c1)
        for (uint32_t k2 = 0; k2 < 16; ++k2) {
            const uint32_t c2 = (k2 + (k2 >= c1 ? 1u : 0u)) & 15u;   // k2 = 15 never occurs (mulhi(w2, 15) < 15)
            for (uint32_t v = 0; v < 4; ++v) {
                uint8_t e[16] = {};
                e[c2] = (uint8_t)(1 + (v & 1));
                e[c1] = (uint8_t)(1 + (v >> 1));
                uint64_t b = 0;
                for (int c = 0; c < 16; ++c) b |= (uint64_t)e[c] << (4 * c);
                s.board[(c1 * 16 + k2) * 4 + v] = Board{(uint32_t)b, (uint32_t)(b >> 32)};
                s.mask[(c1 * 16 + k2) * 4 + v] = (uint8_t)cells_legal_mask(e);
            }
        }
    return s;
}
#if defined(__CUDACC__)
static __constant__ StartTables g_start_tables_dev = make_start_tables();
#endif
static constexpr StartTables g_start_tables_host = make_start_tables();

// reset_board from the Philox words of (gid, t, B2048_DOM_RESET); also returns the board's legal mask
B2_HD Board start_board(const Rand4& w, uint32_t& mask) {
#if defined(__CUDA_ARCH__)
    const StartTables& S = g_start_tables_dev;
#else
    const StartTables& S = g_start_tables_host;
#endif
    const uint32_t i = (mulhi(w.w0, 16u) * 16u + mulhi(w.w2, 15u)) * 4u + (w.w1 >= 0xE6666667u ? 2u : 0u) +
                       (w.w3 >= 0xE6666667u ? 1u : 0u);
    mask = S.mask[i];
    return S.board[i];
}

struct FastTables {
    const uint16_t* left;
    const uint8_t* merge;
    const AggEntry* agg;
    const SelEntry* sel;
    const uint8_t* act;
};

struct FastIO {
    uint32_t lo, hi;            // board in / out
    uint32_t score, step, max_exp;
    uint32_t action;            // in (buffer mode) / out (action played)
    uint32_t mask_in;           // legal mask of the input board (random-legal mode)
    float reward;
    uint32_t flags;
    int32_t merge_sum;
};

// kAct: B2048_ACT_*; kTrack: score / step / max_exp kept (and truncation evaluated)
// step_fast_rnd takes the board's Philox block of (gid, t, B2048_DOM_STEP) from the caller (the fused rollout kernel
// shares it with the policy's sampling word); step_fast computes it.  keys = make_keys(seed) of the env's seed.
// kShaped = false: the caller guarantees empty_tile_reward = merge_reward = endgame_penalty = 0 and bonus off (the env-only
// headline kernel: no instruction spent on them).
template <int kAct, bool kTrack, bool kShaped = true>
B2_HD void step_fast_rnd(FastIO& io, const b2048_env_cfg& cfg, const Rand4& rnd, const PhiloxKeys& keys, uint64_t gid,
                         uint32_t t, const FastTables& T) {

    uint32_t a;
    if (kAct == B2048_ACT_BUFFER) a = io.action & 3u;
    else if (kAct == B2048_ACT_RANDOM_ANY) a = rnd.w2 >> 30;
    else if (kAct == B2048_ACT_PRIORITY) a = pick_priority(io.mask_in & 0xFu, (uint32_t)cfg.action_priority);
    else {
        uint32_t m4 = io.mask_in & 0xFu;
        a = T.act[m4 * 4u + mulhi(rnd.w2, (uint32_t)popc(m4))];
    }
    io.action = a;

    // ---- move: canonicalise, four row lookups, merge statistics, de-canonicalise
    const SelEntry s = T.sel[a];
    uint32_t clo = nib_swap_m(blk_transpose_m(io.lo, s.tm), s.nl, s.nr), chi = nib_swap_m(blk_transpose_m(io.hi, s.tm), s.nl, s.nr);
    uint32_t flo = prmt(clo, chi, s.f_lo), fhi = prmt(clo, chi, s.f_hi);
    uint32_t i0 = flo & 0xFFFFu, i1 = flo >> 16, i2 = fhi & 0xFFFFu, i3 = fhi >> 16;
    uint32_t r0 = T.left[i0], r1 = T.left[i1], r2 = T.left[i2], r3 = T.left[i3];
    const AggEntry g0 = T.agg[T.merge[i0]], g1 = T.agg[T.merge[i1]], g2 = T.agg[T.merge[i2]], g3 = T.agg[T.merge[i3]];
    uint32_t agg = g0.agg + g1.agg + g2.agg + g3.agg;
    uint32_t orm = g0.orm | g1.orm | g2.orm | g3.orm | 1u;   // bit 0 (exponent 0) never merges: msb(orm) is defined
    uint32_t mlo = r0 + (r1 << 16), mhi = r2 + (r3 << 16);
    uint32_t plo = prmt(mlo, mhi, s.i_lo), phi = prmt(mlo, mhi, s.i_hi);
    uint32_t vlo = blk_transpose_m(nib_swap_m(plo, s.nl, s.nr), s.tm), vhi = blk_transpose_m(nib_swap_m(phi, s.nl, s.nr), s.tm);
    const bool changed = ((vlo ^ io.lo) | (vhi ^ io.hi)) != 0u;

    const uint32_t msum = agg & 0xFFFFFu;
    io.merge_sum = (int32_t)msum;
    if (kTrack) {
        io.score += msum;
        io.step += 1u;
    }

    // ---- spawn: k-th empty cell in row-major order via nibble prefix sums (see file header)
    const uint32_t nb_lo = nz8(vlo) >> 3, nb_hi = nz8(vhi) >> 3;   // bit 0 of each nibble: cell occupied
    const uint32_t zb_lo = nb_lo ^ 0x11111111u, zb_hi = nb_hi ^ 0x11111111u;
    const uint32_t P_lo = zb_lo * 0x11111111u, P_hi = zb_hi * 0x11111111u;   // nibble i = #empty among cells 0..i
    const uint32_t c_lo = P_lo >> 28, c_hi = P_hi >> 28;
    const uint32_t n_empty = c_lo + c_hi;
    uint32_t k = mulhi(rnd.w0, n_empty);
    const bool in_hi = k >= c_lo;
    const uint32_t P = in_hi ? P_hi : P_lo;
    k = in_hi ? k - c_lo : k;
    // nibble i of P + (7 - k) * 0x11111111 is P_i + 7 - k <= 15 (P_i <= 8, k <= 7: no carry between nibbles), so its bit 3
    // is set exactly for the cells whose prefix exceeds k
    const uint32_t G = ((P + (7u - k) * 0x11111111u) & 0x88888888u) >> 3;
    const uint32_t iso = G & (0u - G);                                       // 1 << (4 * cell)
    const uint32_t live = (changed && n_empty != 0u) ? 1u : 0u;              // game2048.py:56-58, :110-111
    const uint32_t val = live * (rnd.w1 >= 0xE6666667u ? 2u : 1u);
    const uint32_t ins = iso * val;
    const uint32_t hsel = in_hi ? 0xFFFFFFFFu : 0u;
    uint32_t nlo = vlo | (ins & ~hsel), nhi = vhi | (ins & hsel);

    // ---- legal mask of the new board; occupancy bits reused from the spawn stage
    // N: rows 0,1 at bit 4i, rows 2,3 at bit 4i+1 (the spawned tile's bit: iso times 1 or 2)
    const uint32_t N = nb_lo | (nb_hi * 2u) | (iso * (in_hi ? live * 2u : live));
    const uint32_t MH = 0x03330333u, MV = 0x11113333u;
    const uint32_t Nr = N >> 4;
    const uint32_t EH = (nz8(nlo ^ (nlo >> 4)) >> 3) | (nz8(nhi ^ (nhi >> 4)) >> 2);
    const uint32_t hmerge = ~EH & N & MH;
    const uint32_t left = (~N & Nr & MH) | hmerge;
    const uint32_t right = (N & ~Nr & MH) | hmerge;
    const uint32_t Nd = ((N >> 16) & 0x00003333u) | ((N * 32768u) & 0x11110000u);
    const uint32_t EV = (nz8(nlo ^ funnel_r(nlo, nhi, 16)) >> 3) | (nz8(nhi ^ (nhi >> 16)) >> 2);
    const uint32_t vmerge = ~EV & N & MV;
    const uint32_t up = (~N & Nd & MV) | vmerge;
    const uint32_t down = (N & ~Nd & MV) | vmerge;
    uint32_t mask = (up ? 1u : 0u) | (right ? 2u : 0u) | (down ? 4u : 0u) | (left ? 8u : 0u);
    const bool done = (mask == 0u) & ((nlo | nhi) != 0u);

    // ---- reward (float64 in the reference's order: base * scale, + step_reward)
    const uint32_t max_merged = msb(orm);
    const uint32_t base = cfg.reward_mode == B2048_REWARD_SUM ? msum : ((agg >> 20) & 0xFFu);
    double r = dmul((double)base, cfg.base_reward_scale);
    // shaping terms in the reference's order (env.py:226-259, as in step_one): empty cells of the NEW board (after the
    // spawn), number of merges (agg bits 28..31), new-max-tile bonus, step reward, end-game penalty.  All uniform branches
    // on launch constants; the plain configuration skips them.
    if (kShaped && cfg.empty_tile_reward != 0.0) r = dadd(r, dmul(cfg.empty_tile_reward, (double)(n_empty - live)));
    if (kShaped && cfg.merge_reward != 0.0) r = dadd(r, dmul(cfg.merge_reward, (double)(agg >> 28)));
    if (kTrack && max_merged >= 3u && max_merged > io.max_exp) {                          // env.py:241-250
        io.max_exp = max_merged;
        if (kShaped && cfg.bonus_mode != B2048_BONUS_OFF) {
            const double bonus = cfg.bonus_mode == B2048_BONUS_RAW ? (double)(1u << max_merged) : (double)max_merged;
            r = dadd(r, dmul(bonus, cfg.bonus_scale));
        }
    }
    r = dadd(r, cfg.step_reward);
    if (kShaped && done && cfg.endgame_penalty != 0.0) r = dadd(r, cfg.endgame_penalty);
    io.reward = (float)r;

    bool trunc = false;
    if (kTrack) trunc = cfg.max_steps > 0 && io.step >= (uint32_t)cfg.max_steps && !done;   // env.py:279-286
    uint32_t f = (changed ? B2048_F_CHANGED : 0u) | (done ? B2048_F_DONE : 0u) | (trunc ? B2048_F_TRUNC : 0u) |
                 ((orm >> 16) & 1u ? B2048_F_OVERFLOW : 0u);
    if (cfg.auto_reset && (done | trunc)) {
        const Board nbd = start_board(stream_keyed(keys, gid, t, B2048_DOM_RESET), mask);   // == reset_board(seed, gid, t)
        nlo = nbd.lo; nhi = nbd.hi;
        if (kTrack) { io.score = 0u; io.step = 0u; io.max_exp = 2u; }
    }
    io.lo = nlo; io.hi = nhi;
    io.flags = f | mask;
}

template <int kAct, bool kTrack, bool kShaped = true>
B2_HD void step_fast(FastIO& io, const b2048_env_cfg& cfg, const PhiloxKeys& keys, uint64_t /* seed: carried by keys */,
                     uint64_t gid, uint32_t t, const FastTables& T) {
    step_fast_rnd<kAct, kTrack, kShaped>(io, cfg, stream_keyed(keys, gid, t, B2048_DOM_STEP), keys, gid, t, T);
}
// host side: does this configuration need the shaping terms?
inline bool cfg_is_shaped(const b2048_env_cfg& c) {
    return c.empty_tile_reward != 0.0 || c.merge_reward != 0.0 || c.endgame_penalty != 0.0 || c.bonus_mode != B2048_BONUS_OFF;
}

}  // namespace b2
