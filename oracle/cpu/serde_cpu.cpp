// ORACLE (test / baseline infrastructure, NOT product code): CPU restatement of validated ark-serialize point
// decoding, the rules of oracle/serde.py (de_g1 / de_g2), OpenMP over the elements.  It uses the definition of subgroup
// membership ([r] P = O) and the three-root complex square root, so that it shares no shortcut with the GPU decoders
// (ripp_b200/csrc/serde.cuh).  PARITY UNPINNED against arkworks itself; validated against oracle/serde.py.
// Built on its own (oracle/cpu/serde_binding.py) from the arithmetic of field.hpp / tower.hpp.
#include <omp.h>

#include "tower.hpp"

Fq2 Fq12::FROB1[6];
Fq2 Fq12::FROB2[6];

static const u64 Q_MOD[6] = {0xb9feffffffffaaabull, 0x1eabfffeb153ffffull, 0x6730d2a0f6b0f624ull,
                             0x64774b84f38512bfull, 0x4b1ba7b6434bacd7ull, 0x1a0111ea397fe69aull};
static const u64 R_MOD[4] = {0xffffffff00000001ull, 0x53bda402fffe5bfeull, 0x3339d80809a1d805ull, 0x73eda753299d7d48ull};
static Fq TWO_INV;
static Fq2 B2;  // 4 (1 + u)

template <class F>
struct Aff {
  F x, y;
  bool is_inf() const { return x.is_zero() && y.is_zero(); }
};
// Jacobian (a = 0), the formulas of ark-ec short_weierstrass::Projective
template <class F>
struct Jac {
  F x, y, z;
  static Jac inf() { return {F::one(), F::one(), F::zero()}; }
  bool is_inf() const { return z.is_zero(); }
  Jac dbl() const {
    if (is_inf()) return *this;
    F a = x.sqr(), b = y.sqr(), c = b.sqr();
    F d = ((x + b).sqr() - a - c).dbl();
    F e = a + a.dbl(), f = e.sqr();
    Jac r;
    r.z = (y * z).dbl();
    r.x = f - d.dbl();
    r.y = e * (d - r.x) - c.dbl().dbl().dbl();
    return r;
  }
  Jac add_affine(const Aff<F>& q) const {
    if (q.is_inf()) return *this;
    if (is_inf()) return {q.x, q.y, F::one()};
    F z1z1 = z.sqr(), u2 = q.x * z1z1, s2 = q.y * z * z1z1;
    if (x == u2) {
      if (y == s2) return dbl();
      return inf();
    }
    F h = u2 - x, hh = h.sqr(), i = hh.dbl().dbl(), j = h * i, r = (s2 - y).dbl(), v = x * i;
    Jac o;
    o.x = r.sqr() - j - v.dbl();
    o.y = r * (v - o.x) - (y * j).dbl();
    o.z = (z + h).sqr() - z1z1 - hh;
    return o;
  }
};
// MSB-first double-and-add over a 256-bit canonical scalar
template <class F>
static Jac<F> mul_scalar(const Aff<F>& p, const u64* k) {
  Jac<F> acc = Jac<F>::inf();
  for (int i = 255; i >= 0; i--) {
    acc = acc.dbl();
    if ((k[i / 64] >> (i % 64)) & 1) acc = acc.add_affine(p);
  }
  return acc;
}
static void init_fields() {
  Fq::init(Q_MOD);
  Fr::init(R_MOD);
  TWO_INV = Fq::from_u64(2).inv();
  B2 = {Fq::from_u64(4), Fq::from_u64(4)};
}

// ------------------------------------------------------------------------------------------------
enum { D_OK = 0, D_FLAGS, D_NONCANONICAL, D_NOT_ON_CURVE, D_NOT_IN_SUBGROUP };

static u64 SQRT_EXP[6], HALF[6];  // (p + 1) / 4, (p - 1) / 2
static void init_serde() {
  init_fields();
  u64 t[6];
  memcpy(t, Q_MOD, sizeof(t));
  t[0] += 1;  // p + 1: p is odd, no carry out of limb 0
  for (int i = 0; i < 6; i++) SQRT_EXP[i] = (t[i] >> 2) | (i < 5 ? t[i + 1] << 62 : 0);
  t[0] -= 2;  // p - 1
  for (int i = 0; i < 6; i++) HALF[i] = (t[i] >> 1) | (i < 5 ? t[i + 1] << 63 : 0);
}
// 48 big-endian bytes (top byte masked) -> Montgomery Fq; false if >= p
static bool read_fq(const uint8_t* s, uint8_t top, Fq* out, bool* any) {
  Fq v;
  for (int i = 0; i < 6; i++) {
    u64 w = 0;
    for (int j = 0; j < 8; j++) w = (w << 8) | (u64)(j == 0 && i == 5 ? (s[0] & top) : s[(5 - i) * 8 + j]);
    v.l[i] = w;
    *any = *any || w != 0;
  }
  if (geq<6>(v.l, Q_MOD)) return false;
  *out = v.to_mont();
  return true;
}
static bool lex_largest(const Fq& y) {
  Fq c = y.from_mont();
  return !geq<6>(HALF, c.l);  // c > (p - 1) / 2
}
static bool lex_largest(const Fq2& y) { return y.c1.is_zero() ? lex_largest(y.c0) : lex_largest(y.c1); }
static bool sqrt_fq(const Fq& a, Fq* r) {
  *r = a.pow(SQRT_EXP, 6);
  return r->sqr() == a;
}
static bool sqrt_fq2(const Fq2& a, Fq2* r) {
  Fq s;
  if (a.c1.is_zero()) {
    if (sqrt_fq(a.c0, &s)) {
      *r = {s, Fq::zero()};
      return true;
    }
    if (sqrt_fq(-a.c0, &s)) {
      *r = {Fq::zero(), s};
      return true;
    }
    return false;
  }
  Fq alpha;
  if (!sqrt_fq(a.c0.sqr() + a.c1.sqr(), &alpha)) return false;
  for (int k = 0; k < 2; k++) {
    Fq delta = (k == 0 ? a.c0 + alpha : a.c0 - alpha) * TWO_INV, x0;
    if (!sqrt_fq(delta, &x0) || x0.is_zero()) continue;
    Fq2 y = {x0, a.c1 * x0.dbl().inv()};
    if (y.sqr() == a) {
      *r = y;
      return true;
    }
  }
  return false;
}
static void set_coord(Fq& f, const Fq* v) { f = v[0]; }
static void set_coord(Fq2& f, const Fq* v) { f = {v[1], v[0]}; }
static bool sqrt_any(const Fq& a, Fq* r) { return sqrt_fq(a, r); }
static bool sqrt_any(const Fq2& a, Fq2* r) { return sqrt_fq2(a, r); }
static Fq curve_b(const Fq*) { return Fq::from_u64(4); }
static Fq2 curve_b(const Fq2*) { return B2; }

template <class F>
static int decode_point(const uint8_t* in, bool compressed, Aff<F>* out) {
  constexpr int D = sizeof(F) / sizeof(Fq);
  const int nfq = compressed ? D : 2 * D;
  *out = {F::zero(), F::zero()};
  bool c = in[0] & 0x80, inf = in[0] & 0x40, largest = in[0] & 0x20;
  if (c != compressed || (largest && (!c || inf))) return D_FLAGS;
  Fq v[4];
  bool any = false, canonical = true;
  for (int j = 0; j < nfq; j++) canonical = read_fq(in + 48 * j, j == 0 ? 0x1f : 0xff, &v[j], &any) && canonical;
  if (inf) return any ? D_FLAGS : D_OK;
  if (!canonical) return D_NONCANONICAL;
  F x, y;
  set_coord(x, v);
  F rhs = x.sqr() * x + curve_b(&x);
  if (compressed) {
    if (!sqrt_any(rhs, &y)) return D_NOT_ON_CURVE;
    if (lex_largest(y) != largest) y = -y;
  } else {
    set_coord(y, v + D);
    if (!(y.sqr() == rhs)) return D_NOT_ON_CURVE;
  }
  Aff<F> p{x, y};
  if (!mul_scalar<F>(p, R_MOD).is_inf()) return D_NOT_IN_SUBGROUP;
  *out = p;
  return D_OK;
}
template <class F>
static void decode_all(const uint8_t* in, size_t n, size_t stride, int compressed, Aff<F>* out, uint8_t* status) {
  init_serde();
#pragma omp parallel for schedule(dynamic, 64)
  for (size_t i = 0; i < n; i++) status[i] = (uint8_t)decode_point<F>(in + i * stride, compressed != 0, &out[i]);
}

extern "C" {
int cpu_serde_threads(void) { return omp_get_max_threads(); }
// n elements at `stride` bytes; out = affine Montgomery points (all zero: identity / rejected), status = D_* per element
void cpu_g1_deserialize(const uint8_t* in, size_t n, size_t stride, int compressed, Aff<Fq>* out, uint8_t* status) {
  decode_all<Fq>(in, n, stride, compressed, out, status);
}
void cpu_g2_deserialize(const uint8_t* in, size_t n, size_t stride, int compressed, Aff<Fq2>* out, uint8_t* status) {
  decode_all<Fq2>(in, n, stride, compressed, out, status);
}
}
