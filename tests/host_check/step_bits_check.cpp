// Checks the msb intrinsic of the fast step body (csrc/b2048_device.cuh) against a bit-by-bit scan, compiled with g++.
// Returns the number of mismatches.
#include "../../rl-2048-with-reinforce-and-actor-critic_b200/csrc/b2048_step_fast.cuh"

static uint64_t splitmix(uint64_t& s) {
    uint64_t z = (s += 0x9E3779B97F4A7C15ull);
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

extern "C" {

// msb against a bit-by-bit scan, every single bit and n random non-zero words
int64_t hc_msb_mismatches(int64_t n, uint64_t seed) {
    int64_t bad = 0;
    auto one = [&](uint32_t x) {
        uint32_t ref = 0;
        for (uint32_t b = 0; b < 32; ++b)
            if (x >> b & 1u) ref = b;
        bad += b2::msb(x) != ref;
    };
    for (uint32_t b = 0; b < 32; ++b) one(1u << b);
    uint64_t s = seed;
    for (int64_t i = 0; i < n; ++i) one((uint32_t)(splitmix(s) >> (i & 31)) | 1u);
    return bad;
}

}  // extern "C"
