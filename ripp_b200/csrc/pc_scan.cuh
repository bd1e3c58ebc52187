// The Fr rules of the polynomial-commitment kernels (poly_commit.cuh), host and device, so that a host build
// (tests/hostsim/hostsim_pc.cpp) can check them against the oracle, and the row combination's grouping.
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

static const size_t ROW_THREADS = (size_t)1 << 16;  // threads the row combination aims for (columns x row groups)
static const size_t MAX_ROW_GROUPS = 65535;         // the groups are k_pc_rows' gridDim.y

// G groups of R rows for the row combination of n rows of m (k_pc_rows / k_pc_rows_combine): G m about ROW_THREADS,
// G <= MAX_ROW_GROUPS (only n = 2^16, m = 1 hits the cap: R = 2, G = 2^15), G R >= n > (G - 1) R
RIPP_HD void row_groups(size_t n, size_t m, size_t* G, size_t* R) {
  size_t g = ROW_THREADS / m;
  if (g < 1) g = 1;
  if (g > n) g = n;
  if (g > MAX_ROW_GROUPS) g = MAX_ROW_GROUPS;
  *R = (n + g - 1) / g;
  *G = (n + *R - 1) / *R;
}

// ---- the batched kernels (pc_batch.cuh): count instances of equal shape, instance k's elements at k x its length ----

// instance k and element e of flat index i over segments of `len` elements
RIPP_HD void seg_split(size_t i, size_t len, size_t* k, size_t* e) {
  *k = i / len;
  *e = i - *k * len;
}

// G groups of R rows for the row combination of `count` polynomials of n rows of m (k_pc_rows_seg): G m count about
// ROW_THREADS, G R >= n > (G - 1) R.  The launch is one-dimensional over count G m <= 2^24 threads, so no grid dimension
// caps G (row_blocks).
RIPP_HD void row_groups_batch(size_t count, size_t n, size_t m, size_t* G, size_t* R) {
  size_t g = ROW_THREADS / (m * count);
  if (g < 1) g = 1;
  if (g > n) g = n;
  *R = (n + g - 1) / g;
  *G = (n + *R - 1) / *R;
}

// blocks of 128 threads of k_pc_rows_seg: thread i is column j of group g of instance k, i = (k G + g) m + j
RIPP_HD size_t row_blocks(size_t count, size_t G, size_t m) { return (count * G * m + 127) / 128; }

RIPP_HD void row_index(size_t i, size_t G, size_t m, size_t* k, size_t* g, size_t* j) {
  size_t r;
  seg_split(i, G * m, k, &r);
  seg_split(r, m, g, j);
}

// s^(2^e): the segmented scan's point at level l is z^(L^l) = z^(2^(5 l)) for chunks of L = 32
RIPP_HD Fr pow2k(Fr s, unsigned e) {
  for (unsigned i = 0; i < e; i++) s = s * s;
  return s;
}

// exponent e of a GIPA verifier's final commitment key (gipa.rs:365-399, the order of verify.cuh's final_key_exponents):
// acc times tinv[j] for every bit j set in e, tinv[j] the inverse of transcript element j (last round first)
RIPP_HD Fr key_exponent(const Fr* tinv, size_t e, Fr acc) {
  for (unsigned j = 0; e; j++, e >>= 1)
    if (e & 1) acc = acc * tinv[j];
  return acc;
}

}  // namespace pc
}  // namespace ripp
