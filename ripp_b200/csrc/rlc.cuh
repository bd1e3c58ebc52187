// The scalars of the Groth16 random-linear-combination check (groth16.cu, ripp_groth16_verify_rlc_*), host and device.
//
// r_i is the i-th 16-byte little-endian chunk of the ChaCha20 keystream keyed by the caller's 32-byte seed (hash.h's
// block function, rand_chacha's layout: block b holds r_4b .. r_4b+3), so r_i < 2^128 < r.  The last member of each
// segment then takes 1 - (the sum of the other members' r_i), which makes the segment's scalars sum to one
// (DESIGN.md §4 "Groth16 verification by random linear combination"; oracle: oracle/groth16_rlc.py rlc_scalars).
#pragma once
#include "curve.cuh"
#include "hash.h"

namespace ripp {
namespace rlc {

// r_4b .. r_4b+3 in Montgomery form
RIPP_HD void scalars4(const uint8_t seed[32], uint64_t b, Fr out[4]) {
  uint8_t ks[64];
  ripp_hash::chacha20_block(seed, b, ks);
#pragma unroll
  for (int q = 0; q < 4; q++) {
    Fr f = Fr::zero();
#pragma unroll
    for (int w = 0; w < 4; w++) {
      const uint8_t* p = ks + 16 * q + 4 * w;
      f.v[w] = (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
    }
    out[q] = f.to_mont();
  }
}

// the last member's scalar from the sum of the others'
RIPP_HD Fr last(const Fr& sum_others) { return Fr::one() - sum_others; }

}  // namespace rlc
}  // namespace ripp
