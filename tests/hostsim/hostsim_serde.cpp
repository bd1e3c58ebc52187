// Host-simulation build of ripp_b200/csrc/serde.cuh (TEST INFRASTRUCTURE ONLY): the point decoders the kernels of
// deserialize.cu run, compiled for the host so that tests/test_hostsim_serde.py can compare them with the oracle.
#define RIPP_HOSTSIM 1
#include "../../ripp_b200/csrc/serde.cuh"
#include <string.h>
using namespace ripp;

extern "C" {
// one element; out = packed affine Montgomery words (24 / 48); returns the status
int hs_g1_decode(const uint8_t* in, int compressed, uint32_t* out) {
  G1Aff p;
  int s = compressed ? serde::decode_point<Fq, true>(in, &p) : serde::decode_point<Fq, false>(in, &p);
  memcpy(out, &p, sizeof(p));
  return s;
}
int hs_g2_decode(const uint8_t* in, int compressed, uint32_t* out) {
  G2Aff p;
  int s = compressed ? serde::decode_point<Fq2, true>(in, &p) : serde::decode_point<Fq2, false>(in, &p);
  memcpy(out, &p, sizeof(p));
  return s;
}
int hs_fq2_lex_largest(const uint32_t* y) {
  Fq2 v;
  memcpy(&v, y, sizeof(v));
  return serde::lex_largest(v);
}
int hs_fq2_sqrt(const uint32_t* a, uint32_t* r) {
  Fq2 v, s;
  memcpy(&v, a, sizeof(v));
  bool ok = serde::sqrt(v, &s);
  memcpy(r, &s, sizeof(s));
  return ok;
}
}
