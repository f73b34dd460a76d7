// rng.cuh - the counter RNG of the synthetic inputs (DESIGN.md §9), keyed by (seed, GLOBAL frame, bit, stream).
// Must stay identical to oracle/bp_oracle.c:orc_rng_u64 and tests/oraclelib.py:rng_u64 (the specification).
// Streams in use: 0 BSC flips, 1 simulator messages (csrc/sim.cu), 2 vote-count reads per bit, 3.. vote-count read
// errors, 4 / 5 AWGN Box-Muller (vote counts and AWGN never key the same frame).
#pragma once
#include <cstdint>

namespace dnaldpc {

__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
    z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ULL;
    z ^= z >> 27; z *= 0x94D049BB133111EBULL;
    z ^= z >> 31;
    return z;
}
__host__ __device__ __forceinline__ uint64_t rng_u64(uint64_t seed, uint64_t frame, uint64_t bit, uint64_t stream) {
    uint64_t x = mix64(seed * 0x9E3779B97F4A7C15ULL + frame + 0x632BE59BD9B4E019ULL);
    return mix64(x ^ (bit * 0xD6E8FEB86659FD93ULL + stream * 0xA0761D6478BD642FULL + 0x2545F4914F6CDD1DULL));
}

}  // namespace dnaldpc
