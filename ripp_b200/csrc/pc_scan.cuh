// The Fr rules of the polynomial-commitment kernels (poly_commit.cuh), host and device, so that a host build
// (tests/hostsim/hostsim_pc.cpp) can check them against the oracle.
//
// Division by (X - z) (poly_commit/mod.rs:98-104) is the backward linear recurrence
//   s_N = 0,  s_k = c_k + z s_(k+1)   (k = N-1 .. 0)
// with q_k = s_(k+1) for k < N-1 and f(z) = s_0.  The coefficients are cut into chunks of L; a chunk's head is its
// recurrence started from carry 0 (chunk_head), and the true value at a chunk's start follows from the heads by the
// same recurrence at the point z^L (carry_combine): S_b = head_b + z^L S_(b+1).  A chunk then replays its recurrence
// from the carry S_(b+1) (chunk_replay).
#pragma once
#include <stddef.h>

#include "curve.cuh"

namespace ripp {
namespace pc {

// acc x + c: one step of Horner's rule, and of the recurrence above
RIPP_HD Fr horner_step(const Fr& acc, const Fr& x, const Fr& c) { return acc * x + c; }

// S_b from the chunk's head, z^L and S_(b+1)
RIPP_HD Fr carry_combine(const Fr& head, const Fr& z_pow_l, const Fr& next) { return horner_step(next, z_pow_l, head); }

// s_lo of the recurrence over c[lo, hi) started from s_hi = carry
RIPP_HD Fr chunk_head(const Fr* c, size_t lo, size_t hi, const Fr& z, Fr carry) {
  for (size_t k = hi; k-- > lo;) carry = horner_step(carry, z, c[k]);
  return carry;
}

// the recurrence over c[lo, hi) from s_hi = carry, writing s_k to out0 (k == 0) or out[k - 1]
RIPP_HD void chunk_replay(const Fr* c, size_t lo, size_t hi, const Fr& z, Fr carry, Fr* out0, Fr* out) {
  for (size_t k = hi; k-- > lo;) {
    carry = horner_step(carry, z, c[k]);
    if (k)
      out[k - 1] = carry;
    else
      *out0 = carry;
  }
}

// s^e by square-and-multiply
RIPP_HD Fr pow(Fr s, uint64_t e) {
  Fr acc = Fr::one();
  for (; e; e >>= 1) {
    if (e & 1) acc = acc * s;
    s = s * s;
  }
  return acc;
}

}  // namespace pc
}  // namespace ripp
