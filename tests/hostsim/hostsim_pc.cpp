// Host-simulation build of the polynomial-commitment rules of ripp_b200/csrc/pc_scan.cuh (TEST INFRASTRUCTURE ONLY):
// the chunked division scan of k_pc_div_heads / k_pc_div_replay, driven level by level as div_scan (poly_commit.cuh)
// drives it but with the chunk length L as a parameter, and the row combination's Horner step and grouping, so that
// tests/test_hostsim_pc.py can compare them with the oracle.
#define RIPP_HOSTSIM 1
#include "../../ripp_b200/csrc/pc_scan.cuh"
#include <string.h>

#include <vector>
using namespace ripp;

static void scan(const Fr* c, size_t N, const Fr& z, size_t L, Fr* out0, Fr* out) {
  const size_t nb = (N + L - 1) / L;
  std::vector<Fr> heads(nb), S(nb);
  if (nb > 1) {
    for (size_t b = 0; b < nb; b++) heads[b] = pc::chunk_head(c, b * L, b * L + L < N ? b * L + L : N, z, Fr::zero());
    scan(heads.data(), nb, pc::pow(z, L), L, &S[0], &S[1]);
  }
  for (size_t b = 0; b < nb; b++) {
    size_t hi = b * L + L < N ? b * L + L : N;
    pc::chunk_replay(c, b * L, hi, z, hi < N ? S[b + 1] : Fr::zero(), out0, out);
  }
}

extern "C" {
// q (len - 1 Montgomery Fr) and f(z) (one), as ripp_fr_div_linear_dev computes them with chunks of L
void hs_div_linear(const uint32_t* coeffs, size_t len, const uint32_t* z, size_t L, uint32_t* q, uint32_t* eval) {
  std::vector<Fr> c(len), qq(len ? len - 1 : 0);
  if (len) memcpy(c.data(), coeffs, len * sizeof(Fr));
  Fr zz, ev = Fr::zero();
  memcpy(&zz, z, sizeof(Fr));
  if (len) scan(c.data(), len, zz, L, &ev, qq.data());
  if (!qq.empty()) memcpy(q, qq.data(), qq.size() * sizeof(Fr));
  memcpy(eval, &ev, sizeof(Fr));
}

// carry_combine(head, z^L, next) = head + z^L next
void hs_carry_combine(const uint32_t* head, const uint32_t* zl, const uint32_t* next, uint32_t* out) {
  Fr h, p, n;
  memcpy(&h, head, sizeof(Fr));
  memcpy(&p, zl, sizeof(Fr));
  memcpy(&n, next, sizeof(Fr));
  Fr r = pc::carry_combine(h, p, n);
  memcpy(out, &r, sizeof(Fr));
}

// y[j] = sum_i x^i C[i m + j] (n rows, zeros from len on) with the rows in groups of R recombined with x^R, as
// k_pc_rows / k_pc_rows_combine
void hs_rows(const uint32_t* coeffs, size_t len, size_t m, size_t n, size_t R, const uint32_t* x, uint32_t* y) {
  const Fr* C = (const Fr*)coeffs;
  Fr xx;
  memcpy(&xx, x, sizeof(Fr));
  const size_t G = (n + R - 1) / R;
  const Fr xr = pc::pow(xx, R);
  for (size_t j = 0; j < m; j++) {
    Fr acc = Fr::zero();
    for (size_t g = G; g-- > 0;) {
      Fr part = Fr::zero();
      size_t hi = g * R + R < n ? g * R + R : n;
      for (size_t i = hi; i-- > g * R;) part = pc::horner_step(part, xx, i * m + j < len ? C[i * m + j] : Fr::zero());
      acc = pc::horner_step(acc, xr, part);
    }
    memcpy(y + 8 * j, &acc, sizeof(Fr));
  }
}

// the row combination's G groups of R rows for n rows of m (pc::row_groups, as ripp_pc_open_dev picks them)
void hs_row_groups(size_t n, size_t m, size_t* G, size_t* R) { pc::row_groups(n, m, G, R); }
}
