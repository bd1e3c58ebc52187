// Host-simulation build of the batched polynomial-commitment rules of ripp_b200/csrc/pc_scan.cuh (TEST INFRASTRUCTURE
// ONLY): the segmented row combination of k_pc_rows_seg / k_pc_rows_combine_seg and the segmented division scan of
// k_pc_div_heads_seg / k_pc_div_replay_seg, each thread of a launch run in turn with the same index rules, so that
// tests/test_hostsim_pc_batch.py can compare them with the oracle.
#define RIPP_HOSTSIM 1
#include "../../ripp_b200/csrc/pc_scan.cuh"
#include <string.h>

#include <vector>
using namespace ripp;

// one level of the segmented scan (div_scan_seg with chunks of L): count segments of N at stride N
static void scan_seg(const Fr* c, size_t N, size_t count, const Fr* z, unsigned level, unsigned log_l, Fr* out0, size_t s0, Fr* out,
                     size_t so) {
  const size_t L = (size_t)1 << log_l, nb = (N + L - 1) / L;
  std::vector<Fr> heads(count * nb), S(count * nb);
  if (nb > 1) {
    for (size_t t = 0; t < count * nb; t++) {
      size_t k, b;
      pc::seg_split(t, nb, &k, &b);
      const size_t lo = b * L, hi = lo + L < N ? lo + L : N;
      heads[t] = pc::chunk_head(c + k * N, lo, hi, pc::pow2k(z[k], log_l * level), Fr::zero());
    }
    scan_seg(heads.data(), nb, count, z, level + 1, log_l, S.data(), nb, S.data() + 1, nb);
  }
  for (size_t t = 0; t < count * nb; t++) {
    size_t k, b;
    pc::seg_split(t, nb, &k, &b);
    const size_t lo = b * L, hi = lo + L < N ? lo + L : N;
    pc::chunk_replay(c + k * N, lo, hi, pc::pow2k(z[k], log_l * level), hi < N ? S[t + 1] : Fr::zero(), out0 + k * s0, out + k * so);
  }
}

extern "C" {
// count polynomials of N (>= 1) Montgomery Fr at stride N divided by (X - z_k) with chunks of 2^log_l: quotients at
// stride N (N - 1 each), evaluations at stride 1
void hs_div_batch(const uint32_t* coeffs, size_t count, size_t N, const uint32_t* z, unsigned log_l, uint32_t* q, uint32_t* eval) {
  std::vector<Fr> c(count * N), zz(count), qq(count * N), ev(count);
  memcpy(c.data(), coeffs, c.size() * sizeof(Fr));
  memcpy(zz.data(), z, count * sizeof(Fr));
  scan_seg(c.data(), N, count, zz.data(), 0, log_l, ev.data(), 1, qq.data(), N);
  memcpy(q, qq.data(), qq.size() * sizeof(Fr));
  memcpy(eval, ev.data(), count * sizeof(Fr));
}

// the batched row combination: polynomial k at coeffs + offs[k] with lens[k] coefficients, y (count m Fr) at x_k,
// grouped as pc::row_groups_batch picks it
void hs_rows_batch(const uint32_t* coeffs, const size_t* offs, const size_t* lens, size_t count, size_t n, size_t m, const uint32_t* x,
                   uint32_t* y) {
  const Fr* C = (const Fr*)coeffs;
  const Fr* X = (const Fr*)x;
  size_t G, R;
  pc::row_groups_batch(count, n, m, &G, &R);
  std::vector<Fr> part(count * G * m);
  for (size_t t = 0; t < count * G * m; t++) {
    size_t k, g, j;
    pc::row_index(t, G, m, &k, &g, &j);
    const size_t lo = g * R, hi = lo + R < n ? lo + R : n;
    Fr acc = Fr::zero();
    for (size_t i = hi; i-- > lo;) {
      const size_t at = i * m + j;
      acc = pc::horner_step(acc, X[k], at < lens[k] ? C[offs[k] + at] : Fr::zero());
    }
    part[t] = acc;
  }
  for (size_t t = 0; t < count * m; t++) {
    size_t k, j;
    pc::seg_split(t, m, &k, &j);
    const Fr xr = pc::pow(X[k], R);
    Fr acc = Fr::zero();
    for (size_t g = G; g-- > 0;) acc = pc::horner_step(acc, xr, part[(k * G + g) * m + j]);
    memcpy(y + 8 * t, &acc, sizeof(Fr));
  }
}

void hs_row_groups_batch(size_t count, size_t n, size_t m, size_t* G, size_t* R, size_t* blocks) {
  pc::row_groups_batch(count, n, m, G, R);
  *blocks = pc::row_blocks(count, *G, m);
}

void hs_row_index(size_t i, size_t G, size_t m, size_t* k, size_t* g, size_t* j) { pc::row_index(i, G, m, k, g, j); }
}
