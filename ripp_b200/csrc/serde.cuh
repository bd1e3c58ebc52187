// Validated decoding of ark-serialize 0.4 / ark-bls12-381 0.4 point encodings (SURVEY.md App. A-4), host and device.
//
// Format (ark-bls12-381 0.4 curves/util.rs): coordinates big-endian, 48 bytes per Fq; G1 = x (compressed) or x || y,
// G2 = x.c1 || x.c0 (compressed) or x.c1 || x.c0 || y.c1 || y.c0.  The top three bits of byte 0 are flags:
// 0x80 compressed, 0x40 point at infinity, 0x20 y is the lexicographically largest root.  Checks, in this order
// (an element reports the first that fails; oracle/serde.py states the same rules):
//   FLAGS           compression bit != mode; sort bit without compression or with infinity; infinity with any other bit
//   NONCANONICAL    a coordinate (flag bits masked) >= p
//   NOT_ON_CURVE    y^2 != x^3 + b (uncompressed) / x^3 + b has no square root (compressed)
//   NOT_IN_SUBGROUP the endomorphism tests of in_prime_subgroup below
// Decoded points are affine Montgomery limbs (include/ripp_b200.h); the identity and every rejected element are all
// zero.  Nothing here is secret, so no step needs to run in constant time.
#pragma once
#include "curve.cuh"

namespace ripp {
namespace serde {

enum : uint8_t { OK = 0, FLAGS = 1, NONCANONICAL = 2, NOT_ON_CURVE = 3, NOT_IN_SUBGROUP = 4 };

// 48 big-endian bytes -> 12 little-endian words; `top` masks the first byte (0x1f clears the flags)
RIPP_HD void be48_words(const uint8_t* s, uint32_t* w, uint8_t top) {
#pragma unroll
  for (int i = 0; i < 12; i++) {
    const uint8_t* b = s + 44 - 4 * i;
    w[i] = ((uint32_t)b[0] << 24) | ((uint32_t)b[1] << 16) | ((uint32_t)b[2] << 8) | (uint32_t)b[3];
  }
  w[11] &= ((uint32_t)top << 24) | 0xffffffu;
}

// w < p, as the borrow of w - p
RIPP_HD bool lt_p(const uint32_t* w) {
  uint32_t br = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) {
    uint64_t t = (uint64_t)w[i] - k::FQ_P(i) - br;
    br = (uint32_t)(t >> 63);
  }
  return br != 0;
}

// y > -y for y in Fq: the canonical integer exceeds (p - 1) / 2
RIPP_HD bool lex_largest(const Fq& y) {
  Fq c = y.from_mont();
  uint32_t br = 0;
#pragma unroll
  for (int i = 0; i < 12; i++) {
    uint64_t t = (uint64_t)k::FQ_HALF(i) - c.v[i] - br;
    br = (uint32_t)(t >> 63);
  }
  return br != 0;
}
// ark-ff 0.4 orders Fq2 by c1 first and by c0 only when c1 is equal; y and -y share c1 exactly when c1 = 0
RIPP_HD bool lex_largest(const Fq2& y) { return y.c1.is_zero() ? lex_largest(y.c0) : lex_largest(y.c1); }

// a^((p+1)/4): since p = 3 mod 4 this is a square root of a when a is a square, and of -a otherwise.  Plain
// left-to-right binary powering: no window table to hold in registers.
RIPP_FN Fq fq_pow_sqrt(Fq a) {
  Fq r = Fq::one();
#pragma unroll
  for (int w = 11; w >= 0; w--) {
    const uint32_t e = k::FQ_SQRT_EXP(w);
#pragma unroll 1
    for (int b = 31; b >= 0; b--) {
      r = r.sqr();
      if ((e >> b) & 1) r = r * a;
    }
  }
  return r;
}

RIPP_HD bool sqrt(const Fq& a, Fq* r) {
  *r = fq_pow_sqrt(a);
  return r->sqr() == a;
}

// Complex method.  With alpha^2 = a0^2 + a1^2 and delta = (a0 + alpha) / 2, y = (x, a1 / 2x) for x^2 = delta.  When delta
// is not a square, x = delta^((p+1)/4) satisfies x^2 = -delta, and y = (a1 / 2x, x) is a root instead (expand y^2 with
// alpha^2 - a0^2 = a1^2), so one power serves both cases.  Which of the two roots comes out does not matter: the caller
// normalises the sign.
RIPP_FN bool sqrt(Fq2 a, Fq2* r) {
  if (a.c1.is_zero()) {  // every element of Fq is a square in Fq2: sqrt(a0), or sqrt(-a0) u
    Fq s = fq_pow_sqrt(a.c0);
    *r = s.sqr() == a.c0 ? Fq2{s, Fq::zero()} : Fq2{Fq::zero(), s};
    return true;
  }
  Fq norm = a.c0.sqr() + a.c1.sqr();
  Fq alpha = fq_pow_sqrt(norm);
  if (alpha.sqr() != norm) return false;  // a is a square in Fq2 iff its norm is a square in Fq
  Fq delta = (a.c0 + alpha).half();
  Fq x = fq_pow_sqrt(delta);  // x != 0: delta (a0 - alpha) / 2 = -a1^2 / 4 != 0
  Fq t = a.c1 * x.dbl().inv();
  *r = x.sqr() == delta ? Fq2{x, t} : Fq2{t, x};
  return r->sqr() == a;
}

RIPP_HD void curve_b(Fq& b) {
#pragma unroll
  for (int i = 0; i < 12; i++) b.v[i] = k::G1_B(i);
}
RIPP_HD void curve_b(Fq2& b) {
#pragma unroll
  for (int i = 0; i < 12; i++) {
    b.c0.v[i] = k::G2_B(i);
    b.c1.v[i] = k::G2_B(12 + i);
  }
}

// 48 big-endian bytes -> Fq in Montgomery form (meaningful only when canonical); `any` collects the bits, `canonical`
// whether the value is below p
RIPP_HD Fq load_fq(const uint8_t* s, uint8_t top, uint32_t& any, bool& canonical) {
  Fq f;
  be48_words(s, f.v, top);
#pragma unroll
  for (int i = 0; i < 12; i++) any |= f.v[i];
  canonical = canonical && lt_p(f.v);
  return f.to_mont();
}
// one coordinate in serialised order (G2: c1 first); `first` = it holds the flag bits
RIPP_HD void load_coord(const uint8_t* s, bool first, Fq& f, uint32_t& any, bool& canonical) {
  f = load_fq(s, first ? 0x1f : 0xff, any, canonical);
}
RIPP_HD void load_coord(const uint8_t* s, bool first, Fq2& f, uint32_t& any, bool& canonical) {
  f.c1 = load_fq(s, first ? 0x1f : 0xff, any, canonical);
  f.c0 = load_fq(s + 48, 0xff, any, canonical);
}

// Membership of the prime-order subgroup for a point on the curve (ark-ec is_in_correct_subgroup_assuming_on_curve).
// G1: phi(P) == [x^2 - 1] P, which forces [r] P = O because phi^2 + phi + 1 = 0 on the whole curve and
// lambda^2 + lambda + 1 = r; G2: -psi(P) == [|x|] P.  The scalar multiplications are plain double-and-add: no
// endomorphism is trusted before the test has passed.  The identity is a member.
template <class F>
RIPP_FN bool in_prime_subgroup(const Aff<F>& p) {
  if (p.is_inf()) return true;
  uint32_t bits[4];
  int nbits;
  if (sizeof(F) == sizeof(Fq)) {
#pragma unroll
    for (int j = 0; j < 4; j++) bits[j] = k::ENDO_LAMBDA(j);
    nbits = 128;
  } else {
    bits[0] = (uint32_t)k::X_ABS;
    bits[1] = (uint32_t)(k::X_ABS >> 32);
    bits[2] = bits[3] = 0;
    nbits = 64;
  }
  Jac<F> r = scalar_mul<F>(p, bits, nbits);
  Aff<F> q = endo_map(p);
  F z2 = r.z.sqr();
  return !r.is_inf() && r.x == q.x * z2 && r.y == q.y * z2 * r.z;
}

// One element: `in` holds 48 D (compressed) or 96 D bytes, D = 1 for G1 and 2 for G2.  Returns the status; *out is the
// decoded point, all zero for the identity and for a rejected element.
template <class F, bool COMPRESSED>
RIPP_FN uint8_t decode_point(const uint8_t* in, Aff<F>* out) {
  constexpr int D = sizeof(F) / sizeof(Fq);
  *out = Aff<F>::inf();
  const bool c = in[0] & 0x80, inf = in[0] & 0x40, largest = in[0] & 0x20;
  if (c != COMPRESSED || (largest && (!c || inf))) return FLAGS;
  uint32_t any = 0;
  bool canonical = true;
  F x, y;
  load_coord(in, true, x, any, canonical);
  if (!COMPRESSED) load_coord(in + 48 * D, false, y, any, canonical);
  if (inf) return any ? FLAGS : OK;
  if (!canonical) return NONCANONICAL;
  F b;
  curve_b(b);
  F rhs = x.sqr() * x + b;
  if (COMPRESSED) {
    // get_point_from_x_unchecked: the root y with (y > -y) == the sort flag
    if (!sqrt(rhs, &y)) return NOT_ON_CURVE;
    if (lex_largest(y) != largest) y = -y;
  } else if (y.sqr() != rhs) {
    return NOT_ON_CURVE;
  }
  // tested where it is stored: nothing of this frame stays live across the subgroup test
  *out = Aff<F>{x, y};
  if (in_prime_subgroup(*out)) return OK;
  *out = Aff<F>::inf();
  return NOT_IN_SUBGROUP;
}

}  // namespace serde
}  // namespace ripp
