// Host-simulation build of the public-input rule of ripp_b200/csrc/serde.cuh (TEST INFRASTRUCTURE ONLY): the
// per-element decode k_fr_deserialize runs, compiled for the host so that tests/test_hostsim_groth16.py can compare it
// with the oracle.
#define RIPP_HOSTSIM 1
#include "../../ripp_b200/csrc/serde.cuh"
#include <string.h>
using namespace ripp;

extern "C" {
// one element; out = 8 Montgomery words (zero when rejected); returns 1 for a canonical element
int hs_fr_decode(const uint8_t* in, uint32_t* out) {
  Fr f;
  bool ok = serde::decode_fr(in, &f);
  memcpy(out, &f, sizeof(f));
  return ok;
}
}
