// np_rng_check.cpp — TEST INFRASTRUCTURE.  Compiles the product's NumPy-stream header (b2048_np_rng.cuh, host+device)
// with g++ so that tests/test_np_streams.py can compare it with the installed NumPy without a GPU.
// A generator state crosses the boundary as six uint64: state_hi, state_lo, inc_hi, inc_lo, has_uint32, uinteger.
#include <cstdint>
#include "../../rl-2048-with-reinforce-and-actor-critic_b200/csrc/b2048_np_rng.cuh"

static b2048_np_rng load(const uint64_t* w) {
    b2048_np_rng r;
    r.state_hi = w[0]; r.state_lo = w[1]; r.inc_hi = w[2]; r.inc_lo = w[3];
    r.has_uint32 = (uint32_t)w[4]; r.uinteger = (uint32_t)w[5]; r.reserved = 0;
    return r;
}

static void store(const b2048_np_rng& r, uint64_t* w) {
    w[0] = r.state_hi; w[1] = r.state_lo; w[2] = r.inc_hi; w[3] = r.inc_lo; w[4] = r.has_uint32; w[5] = r.uinteger;
}

extern "C" {

int npc_sizeof_rng() { return (int)sizeof(b2048_np_rng); }

void npc_seed(const uint64_t* seeds, uint64_t* out, int64_t n) {
    for (int64_t i = 0; i < n; ++i) store(b2::np::seed(seeds[i]), out + 6 * i);
}

// ops[i]: 0 = integers(arg[i]), 1 = random(), 2 = choice(4, p = probs[4i .. 4i+3]), 3 = spawn_draw(arg[i]) (k | four << 4)
void npc_run(uint64_t* state, const int32_t* ops, const uint32_t* arg, const float* probs, double* out, int64_t n) {
    b2048_np_rng r = load(state);
    for (int64_t i = 0; i < n; ++i) {
        switch (ops[i]) {
            case 0: out[i] = (double)b2::np::bounded(r, arg[i]); break;
            case 1: out[i] = b2::np::next_double(r); break;
            case 2: out[i] = (double)b2::np::choice4(r, probs[4 * i], probs[4 * i + 1], probs[4 * i + 2], probs[4 * i + 3]); break;
            default: out[i] = (double)b2::np::spawn_draw(r, arg[i]); break;
        }
    }
    store(r, state);
}

// Game2048._spawn on packed boards (in place) and Game2048.reset boards, each from its own stream (advanced in place)
void npc_spawn(uint64_t* states, uint64_t* boards, int64_t n) {
    for (int64_t i = 0; i < n; ++i) {
        b2048_np_rng r = load(states + 6 * i);
        boards[i] = b2::to_u64(b2::np::spawn(r, b2::make_board(boards[i])));
        store(r, states + 6 * i);
    }
}

void npc_reset(uint64_t* states, uint64_t* boards, int64_t n) {
    for (int64_t i = 0; i < n; ++i) {
        b2048_np_rng r = load(states + 6 * i);
        boards[i] = b2::to_u64(b2::np::reset_board(r));
        store(r, states + 6 * i);
    }
}

}  // extern "C"
