// Host-simulation build of the final-key exponent rule of ripp_b200/csrc/pc_scan.cuh (TEST INFRASTRUCTURE ONLY): the
// index rule of k_pc_key_exponents_seg (pc_verify_batch.cuh), each thread of a launch run in turn, so that
// tests/test_hostsim_pc_verify_batch.py can compare it with the oracle's final commitment keys.
#define RIPP_HOSTSIM 1
#include "../../ripp_b200/csrc/pc_scan.cuh"
#include <string.h>

using namespace ripp;

extern "C" {
// k_pc_key_exponents_seg: count exponent vectors of 2^L Fr from count x L inverses, times factor[k] (NULL: one)
void hs_key_exponents(const uint32_t* tinv, unsigned L, const uint32_t* factor, size_t count, uint32_t* out) {
  const size_t len = (size_t)1 << L;
  const Fr* T = (const Fr*)tinv;
  const Fr* F = (const Fr*)factor;
  for (size_t t = 0; t < count * len; t++) {
    size_t k, e;
    pc::seg_split(t, len, &k, &e);
    const Fr v = pc::key_exponent(T + k * L, e, F ? F[k] : Fr::one());
    memcpy(out + 8 * t, &v, sizeof(Fr));
  }
}
}
