// Scalar decomposition for the endomorphism-accelerated scalar multiplications (host and device).
//   G1: c = d0 + d1 lambda,           lambda = x^2 - 1 (128 bits), E = phi  = [lambda]
//   G2: c = d0 + d1 B + d2 B^2 + d3 B^3,   B = |x| (64 bits),      E = -psi = [|x|]
// so  c P = sum_i d_i E^i(P): a joint double-and-add over max |d_i| bits.  Digits are NAF-recoded into
// +1 / -1 bitmaps.  (curve.cuh: endo_map; eigenvalues checked in tests/test_hostsim.py::test_endomorphisms.)
#pragma once
#include "curve.cuh"

namespace ripp {

struct EndoBits {
  uint32_t pos[4][5], neg[4][5];
  int m, nbits;
};

// NAF of a little-endian `words`-word integer: digit i = +1 / -1 / 0 by bit i of pos / neg
RIPP_HD void naf_bitmaps(const uint32_t* k_in, int words, uint32_t* pos, uint32_t* neg, int* nd) {
  uint32_t k[6];
  for (int i = 0; i < 6; i++) k[i] = i < words ? k_in[i] : 0u;
  int i = 0;
  for (; i < 160; i++) {
    uint32_t any = 0;
    for (int j = 0; j < 6; j++) any |= k[j];
    if (!any) break;
    if (k[0] & 1) {
      if ((k[0] & 3) == 1) {
        pos[i >> 5] |= 1u << (i & 31);
        k[0] -= 1;
      } else {
        neg[i >> 5] |= 1u << (i & 31);
        uint32_t carry = 1;
        for (int j = 0; j < 6; j++) {
          uint32_t t = k[j] + carry;
          carry = (t < carry) ? 1u : 0u;
          k[j] = t;
        }
      }
    }
    for (int j = 0; j < 5; j++) k[j] = (k[j] >> 1) | (k[j + 1] << 31);
    k[5] >>= 1;
  }
  *nd = i;
}

// (q, r) = divmod(k, d): k, q 8 words; d, r `dw` <= 4 words.  Bitwise restoring division: ~5 k cheap
// instructions, negligible next to the ~10^6 of the scalar multiplication it shortens.
RIPP_HD void divmod_words(const uint32_t* k, const uint32_t* d, int dw, uint32_t* q, uint32_t* r) {
  uint32_t rem[5] = {0, 0, 0, 0, 0};
  for (int i = 0; i < 8; i++) q[i] = 0;
  for (int bit = 255; bit >= 0; bit--) {
    for (int j = 4; j > 0; j--) rem[j] = (rem[j] << 1) | (rem[j - 1] >> 31);
    rem[0] = (rem[0] << 1) | ((k[bit >> 5] >> (bit & 31)) & 1);
    bool ge = true, decided = false;
    for (int j = 4; j >= 0; j--) {
      uint32_t dj = j < dw ? d[j] : 0u;
      if (!decided && rem[j] != dj) {
        ge = rem[j] > dj;
        decided = true;
      }
    }
    if (ge) {
      uint32_t borrow = 0;
      for (int j = 0; j < 5; j++) {
        uint32_t dj = j < dw ? d[j] : 0u;
        uint32_t t = rem[j] - dj - borrow;
        borrow = (rem[j] < dj || (rem[j] == dj && borrow)) ? 1u : 0u;
        rem[j] = t;
      }
      q[bit >> 5] |= 1u << (bit & 31);
    }
  }
  for (int j = 0; j < dw; j++) r[j] = rem[j];
}

// digits of a canonical (non-Montgomery) scalar; GROUP = 1 for G1, 2 for G2
template <int GROUP>
RIPP_HD void endo_digits(const uint32_t* canon, uint32_t digits[4][4], int* m) {
  uint32_t base[4] = {0, 0, 0, 0};
  int bw;
  if (GROUP == 1) {
    for (int i = 0; i < 4; i++) base[i] = k::ENDO_LAMBDA(i);
    bw = 4;
  } else {
    base[0] = (uint32_t)k::X_ABS;
    base[1] = (uint32_t)(k::X_ABS >> 32);
    bw = 2;
  }
  // exactly MAXD digits: the last one takes the whole remaining quotient (c < r = lambda^2 + lambda + 1 gives
  // d1 <= lambda + 1 < 2^128 on G1; c < r < |x|^4 gives d3 < |x| on G2), so no higher power of E is ever needed
  const int MAXD = GROUP == 1 ? 2 : 4;
  uint32_t cur[8], q[8];
  for (int i = 0; i < 8; i++) cur[i] = canon[i];
  *m = 0;
  for (int i = 0; i < 4; i++) {
    for (int j = 0; j < 4; j++) digits[i][j] = 0;
    if (i >= MAXD) continue;
    uint32_t any = 0;
    for (int j = 0; j < 8; j++) any |= cur[j];
    if (!any) continue;
    if (i == MAXD - 1) {
      for (int j = 0; j < 4; j++) digits[i][j] = cur[j];
      for (int j = 0; j < 8; j++) cur[j] = 0;
    } else {
      divmod_words(cur, base, bw, q, digits[i]);
      for (int j = 0; j < 8; j++) cur[j] = q[j];
    }
    *m = i + 1;
  }
}

template <int GROUP>
RIPP_HD void endo_decompose(const uint32_t* canon, EndoBits& b) {
  for (int i = 0; i < 4; i++)
    for (int j = 0; j < 5; j++) b.pos[i][j] = b.neg[i][j] = 0;
  uint32_t digits[4][4];
  endo_digits<GROUP>(canon, digits, &b.m);
  b.nbits = 0;
  for (int i = 0; i < b.m; i++) {
    int nd = 0;
    naf_bitmaps(digits[i], 4, b.pos[i], b.neg[i], &nd);
    if (nd > b.nbits) b.nbits = nd;
  }
}

// Split recoding for the fold with precomputed bases (msm.cu: k_fold_pre, k_fold4_xp<true>): the NAF of digit k is cut at
// bit H, digits below H stay on E^k(P) and digits at H and above go to E^k(D), D = [2^H] P, at position j - H.  Cutting the
// NAF rather than the integer keeps the sum exact when the recoding carries past bit H.  Part 2k + s holds the low (s = 0)
// or high (s = 1) half of digit k: G1 (H = 64) four parts of <= 65 digits, G2 (H = 32) eight parts of <= 33 digits, so
// the chain of a part is half of what it walks without D.
template <int GROUP>
struct SplitOf {
  static constexpr int H = GROUP == 1 ? 64 : 32;
  static constexpr int PARTS = GROUP == 1 ? 4 : 8;  // 2 x endo_digits' MAXD
};
struct EndoSplit {
  uint32_t pos[8][3], neg[8][3];
  int nbits[8];  // digits of each part
};

template <int GROUP>
RIPP_HD void endo_split(const EndoBits& b, EndoSplit& s) {
  constexpr int H = SplitOf<GROUP>::H;
  for (int t = 0; t < 8; t++) {
    s.nbits[t] = 0;
    for (int w = 0; w < 3; w++) s.pos[t][w] = s.neg[t][w] = 0;
  }
  for (int k = 0; k < SplitOf<GROUP>::PARTS / 2; k++)
    for (int j = 0; j < 160; j++) {
      const bool ps = (b.pos[k][j >> 5] >> (j & 31)) & 1, ng = (b.neg[k][j >> 5] >> (j & 31)) & 1;
      if (!(ps || ng)) continue;
      const int t = 2 * k + (j >= H), i = j >= H ? j - H : j;  // i < 96: a digit's NAF has at most 129 positions
      (ps ? s.pos : s.neg)[t][i >> 5] |= 1u << (i & 31);
      if (i + 1 > s.nbits[t]) s.nbits[t] = i + 1;
    }
}

// Same sum when every lane of a warp has its OWN scalar: one addition slot per (bit, digit) whose operand is
// selected (+base, -base or the identity), so the warp runs the addition body once per slot instead of once per
// distinct sign pattern.
template <class F>
RIPP_FN Jac<F> endo_mul_simt(const Aff<F>& p, const EndoBits& c, int m_uniform, int nbits_uniform) {
  Aff<F> base[4];
  base[0] = p;
  for (int t = 1; t < m_uniform; t++) base[t] = endo_map(base[t - 1]);
  Jac<F> acc = Jac<F>::inf();
  for (int j = nbits_uniform - 1; j >= 0; j--) {
    acc = acc.dbl();
    for (int t = 0; t < m_uniform; t++) {
      bool ps = (c.pos[t][j >> 5] >> (j & 31)) & 1, ng = (c.neg[t][j >> 5] >> (j & 31)) & 1;
      Aff<F> q = base[t];
      if (ng) q = q.neg();
      if (!(ps || ng)) q = Aff<F>::inf();
      acc = acc.add_mixed(q);
    }
  }
  return acc;
}

// sum_i d_i E^i(p) as a Jacobian point
template <class F>
RIPP_FN Jac<F> endo_mul(const Aff<F>& p, const EndoBits& c) {
  Aff<F> base[4];
  base[0] = p;
  for (int t = 1; t < c.m; t++) base[t] = endo_map(base[t - 1]);
  Jac<F> acc = Jac<F>::inf();
  for (int j = c.nbits - 1; j >= 0; j--) {
    acc = acc.dbl();
    for (int t = 0; t < c.m; t++) {
      if ((c.pos[t][j >> 5] >> (j & 31)) & 1) acc = acc.add_mixed(base[t]);
      if ((c.neg[t][j >> 5] >> (j & 31)) & 1) acc = acc.add_mixed(base[t].neg());
    }
  }
  return acc;
}

}  // namespace ripp
