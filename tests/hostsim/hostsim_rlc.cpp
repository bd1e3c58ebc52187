// Host-simulation build of the scalar rules of ripp_b200/csrc/rlc.cuh (TEST INFRASTRUCTURE ONLY): the ChaCha20 block
// of hash.h and the scalar derivation k_rlc_scalars / k_rlc_segment_fr run, compiled for the host so that
// tests/test_hostsim_rlc.py can compare them with the oracle.
#define RIPP_HOSTSIM 1
#include "../../ripp_b200/csrc/rlc.cuh"
#include <string.h>
using namespace ripp;

extern "C" {
void hs_chacha20_block(const uint8_t* key, uint64_t counter, uint8_t* out) { ripp_hash::chacha20_block(key, counter, out); }

// r_4b .. r_4b+3: 32 Montgomery words
void hs_rlc_scalars4(const uint8_t* seed, uint64_t b, uint32_t* out) {
  Fr r[4];
  rlc::scalars4(seed, b, r);
  memcpy(out, r, sizeof(r));
}

// one segment's normalisation as the kernels do it: r (k Montgomery scalars, members first to last) -> the last
// member's scalar, 1 - the others' sum
void hs_rlc_last(const uint32_t* r, uint32_t k, uint32_t* out) {
  Fr acc = Fr::zero();
  for (uint32_t i = 0; i + 1 < k; i++) {
    Fr v;
    memcpy(&v, r + 8 * i, sizeof(v));
    acc = acc + v;
  }
  Fr l = rlc::last(acc);
  memcpy(out, &l, sizeof(l));
}
}
