// "xt": lane teams for the latency-bound point kernels -- the folds A' = A_R c + A_L / v' = v_R c^-1 + v_L of the
// late GIPA rounds (gipa.rs:261-291; mul_helper, ip_proofs/src/lib.rs:15-19) and the normalisations behind them.
//
// One curve point is handled by a TEAM OF LANES OF ONE WARP: 3 lanes for G1 (coordinates in Fq), 9 lanes for G2
// (coordinates in Fq2: 3 product units x 3 Karatsuba roles).  The point formulas are written as LEVELS of up to
// three independent field products (dbl-2009-l: 3 levels, madd-2007-bl: 5 levels); in a level every lane of the
// team computes exactly ONE Fq Montgomery product, the results are exchanged through the team's slice of shared
// memory, and every lane of the team carries the identical point state in registers.  Field additions between the
// levels are recomputed by all lanes of the team (same instruction stream: no extra time).
//
// Why lanes: a warp instruction occupies the multiplier pipe for the same time whatever the number of active lanes,
// and the vectors of the late rounds are short (n' <= 512 elements = 171 warps of G2 teams for 592 sub-partitions),
// so the length of ONE element's dependent chain is the whole cost: 7 / 11 Fq2-product levels per doubling / addition
// on one lane's stream (3 Fq products each) become 3 / 5 levels of one Fq product.  x3.cuh (teams of three WARPS,
// one lane per element) remains for vectors long enough to fill the sub-partitions.
#pragma once
#include "endo.cuh"

namespace ripp {
namespace xt {

template <class F>
struct TeamOf;
template <>
struct TeamOf<Fq> {
  static constexpr int LANES = 3;          // one Fq product per lane and level
  static constexpr int PER_WARP = 10;      // lanes 30, 31 mirror lanes 0, 1
  static constexpr int BUS_WORDS = 3 * 12; // per buffer
};
template <>
struct TeamOf<Fq2> {
  static constexpr int LANES = 9;          // unit u = t / 3 (which product of the level), role r = t % 3 (Karatsuba part)
  static constexpr int PER_WARP = 3;       // lanes 27..31 mirror lanes 0..4
  static constexpr int BUS_WORDS = 9 * 12;
};

struct Team {
  int t;             // lane within the team
  uint32_t* bus;     // 2 buffers of BUS_WORDS words (alternated: one barrier per exchange, see l6.cuh gather3)
  mutable int par;
  void* bar;         // host build: barrier of the team's threads
};

#if defined(__CUDA_ARCH__)
__device__ __forceinline__ void sync(const Team&) { __syncwarp(); }
#else
void host_barrier(void* bar);
inline void sync(const Team& tm) { host_barrier(tm.bar); }
#endif

RIPP_HD Fq fqmul(const Fq& a, const Fq& b) { return Fq::mul_fn(a, b); }
RIPP_HD Fq sel3(int r, const Fq& a, const Fq& b, const Fq& c) {
  Fq o;
#pragma unroll
  for (int i = 0; i < 12; i++) o.v[i] = r == 0 ? a.v[i] : (r == 1 ? b.v[i] : c.v[i]);
  return o;
}
RIPP_HD Fq2 sel3(int r, const Fq2& a, const Fq2& b, const Fq2& c) { return {sel3(r, a.c0, b.c0, c.c0), sel3(r, a.c1, b.c1, c.c1)}; }
RIPP_HD void bus_st(uint32_t* p, const Fq& a) {
#if defined(__CUDA_ARCH__)
  uint4* q = reinterpret_cast<uint4*>(p);
#pragma unroll
  for (int i = 0; i < 3; i++) q[i] = make_uint4(a.v[4 * i], a.v[4 * i + 1], a.v[4 * i + 2], a.v[4 * i + 3]);
#else
  for (int i = 0; i < 12; i++) p[i] = a.v[i];
#endif
}
RIPP_HD Fq bus_ld(const uint32_t* p) {
  Fq r;
#if defined(__CUDA_ARCH__)
  const uint4* q = reinterpret_cast<const uint4*>(p);
#pragma unroll
  for (int i = 0; i < 3; i++) {
    uint4 v = q[i];
    r.v[4 * i] = v.x;
    r.v[4 * i + 1] = v.y;
    r.v[4 * i + 2] = v.z;
    r.v[4 * i + 3] = v.w;
  }
#else
  for (int i = 0; i < 12; i++) r.v[i] = p[i];
#endif
  return r;
}

// One level: p_j = u_j * v_j, j = 0, 1, 2, computed by the team; every lane returns all three products.
RIPP_HD void mul3(const Team& tm, const Fq& u0, const Fq& v0, const Fq& u1, const Fq& v1, const Fq& u2, const Fq& v2, Fq& p0,
                  Fq& p1, Fq& p2) {
  uint32_t* b = tm.bus + tm.par * TeamOf<Fq>::BUS_WORDS;
  tm.par ^= 1;
  bus_st(b + tm.t * 12, fqmul(sel3(tm.t, u0, u1, u2), sel3(tm.t, v0, v1, v2)));
  sync(tm);
  p0 = bus_ld(b);
  p1 = bus_ld(b + 12);
  p2 = bus_ld(b + 24);
}
RIPP_HD void mul3(const Team& tm, const Fq2& u0, const Fq2& v0, const Fq2& u1, const Fq2& v1, const Fq2& u2, const Fq2& v2,
                  Fq2& p0, Fq2& p1, Fq2& p2) {
  uint32_t* b = tm.bus + tm.par * TeamOf<Fq2>::BUS_WORDS;
  uint32_t* b2 = tm.bus + (tm.par ^ 1) * TeamOf<Fq2>::BUS_WORDS;  // two exchanges per level: the parity is unchanged after it
  const int u = tm.t / 3, r = tm.t % 3;
  Fq2 x = sel3(u, u0, u1, u2), y = sel3(u, v0, v1, v2);
  // Karatsuba part r of x * y; the cross operands stay unreduced (< 2p each: the product is < 4 p^2 / R + p < 2p,
  // which its final subtraction handles)
  Fq sx, sy;
  {
    using namespace limb;
    add_cc(sx.v[0], x.c0.v[0], x.c1.v[0]);
#pragma unroll
    for (int i = 1; i < 11; i++) addc_cc(sx.v[i], x.c0.v[i], x.c1.v[i]);
    addc(sx.v[11], x.c0.v[11], x.c1.v[11]);
    add_cc(sy.v[0], y.c0.v[0], y.c1.v[0]);
#pragma unroll
    for (int i = 1; i < 11; i++) addc_cc(sy.v[i], y.c0.v[i], y.c1.v[i]);
    addc(sy.v[11], y.c0.v[11], y.c1.v[11]);
  }
  bus_st(b + tm.t * 12, fqmul(sel3(r, x.c0, x.c1, sx), sel3(r, y.c0, y.c1, sy)));
  sync(tm);
  // Second exchange: lane t < 6 recombines ONE component of one product (lanes 6..8 repeat lanes 0..2) instead of
  // every lane recombining all six -- nine modular subtractions on each lane's chain become two.
  {
    const int t6 = tm.t % 6, j = t6 >> 1;
    const bool c1 = t6 & 1;
    const uint32_t* q = b + (3 * j) * 12;
    Fq t0 = bus_ld(q), t1 = bus_ld(q + 12), t2 = bus_ld(q + 24);
    Fq d = sel3(c1 ? 1 : 0, t0, t2, t2) - t1;
    Fq e = d - t0;
    if (tm.t < 6) bus_st(b2 + t6 * 12, sel3(c1 ? 1 : 0, d, e, e));
  }
  sync(tm);
  p0 = {bus_ld(b2), bus_ld(b2 + 12)};
  p1 = {bus_ld(b2 + 24), bus_ld(b2 + 36)};
  p2 = {bus_ld(b2 + 48), bus_ld(b2 + 60)};
}

// dbl-2009-l in three levels; the identity (Z = 0) maps to itself
template <class F>
RIPP_HD Jac<F> dbl(const Team& tm, const Jac<F>& p) {
  F A, B, YZ, C, T, Fv, M, d0, d1;
  mul3(tm, p.x, p.x, p.y, p.y, p.y, p.z, A, B, YZ);
  F E = A.dbl() + A, XB = p.x + B;
  mul3(tm, B, B, XB, XB, E, E, C, T, Fv);
  F D = (T - A - C).dbl();
  Jac<F> r;
  r.x = Fv - D.dbl();
  r.z = YZ.dbl();
  mul3(tm, E, D - r.x, E, E, E, E, M, d0, d1);
  r.y = M - C.dbl().dbl().dbl();
  return r;
}
// madd-2007-bl in five levels, executed unconditionally (every lane reaches every exchange); teams in an
// exceptional case (either operand the identity, P = +-Q) then recompute with the complete single-thread formulas
template <class F>
RIPP_HD Jac<F> madd(const Team& tm, const Jac<F>& p, const Aff<F>& q) {
  F Z1Z1, YZ, d0, U2, S2, HH, ZH2, RR, J, V, YJ, M;
  mul3(tm, p.z, p.z, q.y, p.z, p.z, p.z, Z1Z1, YZ, d0);
  mul3(tm, q.x, Z1Z1, YZ, Z1Z1, q.x, Z1Z1, U2, S2, d0);
  F H = U2 - p.x;
  F rr = (S2 - p.y).dbl();
  F ZH = p.z + H;
  mul3(tm, H, H, ZH, ZH, rr, rr, HH, ZH2, RR);
  F I = HH.dbl().dbl();
  mul3(tm, H, I, p.x, I, H, I, J, V, d0);
  Jac<F> r;
  r.x = RR - J - V.dbl();
  r.z = ZH2 - Z1Z1 - HH;
  mul3(tm, rr, V - r.x, p.y, J, p.y, J, M, YJ, d0);
  r.y = M - YJ.dbl();
  if (q.is_inf() || p.is_inf() || H.is_zero()) return p.add_mixed_body(q);
  return r;
}

// a^-1 for the normalisation: Fq directly; Fq2 through the norm (conj(a) / (c0^2 + c1^2)), every lane redundantly
RIPP_HD Fq inv(const Fq& a) { return a.inv(); }
RIPP_HD Fq2 inv(const Fq2& a) { return a.inv(); }
// affine form without the identity's early exit (Z = 0 inverts to 0, which gives (0, 0) = the packed identity)
template <class F>
RIPP_HD Aff<F> to_affine(const Team& tm, const Jac<F>& a) {
  F zi = inv(a.z), zi2, zi3, x, y, d0, d1;
  mul3(tm, zi, zi, zi, zi, zi, zi, zi2, d0, d1);
  mul3(tm, a.x, zi2, zi2, zi, zi2, zi, x, zi3, d0);
  mul3(tm, a.y, zi3, a.y, zi3, a.y, zi3, y, d0, d1);
  return {x, y};
}

// word-wise copies of a packed affine point to / from the team's scratch
template <class F>
RIPP_HD void aff_st(uint32_t* p, const Aff<F>& a) {
  const uint32_t* w = reinterpret_cast<const uint32_t*>(&a);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(Aff<F>) / 4); i++) p[i] = w[i];
}
template <class F>
RIPP_HD Aff<F> aff_ld(const uint32_t* p) {
  Aff<F> a;
  uint32_t* w = reinterpret_cast<uint32_t*>(&a);
#pragma unroll
  for (int i = 0; i < (int)(sizeof(Aff<F>) / 4); i++) w[i] = p[i];
  return a;
}

// sum_i d_i E^i(p) (endo.cuh) with the team's formulas; control flow depends only on the SHARED scalar.
// `bases`: 4 * sizeof(Aff<F>) / 4 words of the team's scratch for p, E(p), E^2(p), E^3(p) (kept out of the registers:
// the accumulator and the temporaries of an addition already fill them).
// (all of it inlined into the one kernel that uses it: 72-word Jacobian operands of an out-of-line call would travel
// through local memory, x3.cuh measured 20 % of the instructions that way)
template <class F>
RIPP_HD Jac<F> endo_mul(const Team& tm, const Aff<F>& p, const EndoBits& c, uint32_t* bases) {
  constexpr int AW = sizeof(Aff<F>) / 4;
  {
    Aff<F> b = p;
    for (int t = 0; t < c.m; t++) {
      if (tm.t == 0) aff_st<F>(bases + t * AW, b);
      if (t + 1 < c.m) b = endo_map(b);
    }
  }
  sync(tm);
  Jac<F> acc = Jac<F>::inf();
#pragma unroll 1
  for (int j = c.nbits - 1; j >= 0; j--) {
    acc = dbl<F>(tm, acc);
#pragma unroll 1
    for (int t = 0; t < c.m; t++) {
      const bool ps = (c.pos[t][j >> 5] >> (j & 31)) & 1, ng = (c.neg[t][j >> 5] >> (j & 31)) & 1;
      if (ps || ng) {  // one call site: the addition body is instantiated once
        Aff<F> q = aff_ld<F>(bases + t * AW);
        if (ng) q = q.neg();
        acc = madd<F>(tm, acc, q);
      }
    }
  }
  return acc;
}

// d_part E^part(p) alone: the part-parallel fold gives every endomorphism part of an element its own team (in its own
// warp: the bit pattern of a part is the warp's control flow) and adds the parts afterwards, so the dependent chain of
// an element is one 64-bit (G2) / 128-bit (G1) double-and-add instead of four / two interleaved ones.
// `base`: sizeof(Aff<F>) / 4 words of the team's scratch.
// d E^k(p) for one NAF digit set d (`nbits` digits in the bitmaps pos / neg): the chain of one part.
template <class F>
RIPP_HD Jac<F> naf_mul_endo(const Team& tm, const Aff<F>& p, int m, int k, const uint32_t* pos, const uint32_t* neg, int nbits,
                            uint32_t* base) {
  constexpr int AW = sizeof(Aff<F>) / 4;
  {
    // every lane walks the whole chain p, E(p), E^2(p), ... and keeps the image of its part (word-wise select)
    // (m = the group's full part count: parts the scalar does not reach have empty bit patterns and give the identity)
    Aff<F> b = p, mine = p;
    for (int t = 1; t < m; t++) {
      b = endo_map(b);
      uint32_t* mw = reinterpret_cast<uint32_t*>(&mine);
      const uint32_t* bw = reinterpret_cast<const uint32_t*>(&b);
#pragma unroll
      for (int i = 0; i < AW; i++) mw[i] = t == k ? bw[i] : mw[i];
    }
    if (tm.t == 0) aff_st<F>(base, mine);
  }
  sync(tm);
  Jac<F> acc = Jac<F>::inf();
#pragma unroll 1
  for (int j = nbits - 1; j >= 0; j--) {
    acc = dbl<F>(tm, acc);
    const bool ps = (pos[j >> 5] >> (j & 31)) & 1, ng = (neg[j >> 5] >> (j & 31)) & 1;
    if (ps || ng) {
      Aff<F> q = aff_ld<F>(base);
      if (ng) q = q.neg();
      acc = madd<F>(tm, acc, q);
    }
  }
  return acc;
}
template <class F>
RIPP_HD Jac<F> part_mul(const Team& tm, const Aff<F>& p, const EndoBits& c, int m, int part, uint32_t* base) {
  return naf_mul_endo<F>(tm, p, m, part, c.pos[part], c.neg[part], c.nbits, base);
}

// [2^h] p in affine form: the base D of the split recoding's high parts (endo.cuh: endo_split); the identity stays the identity
template <class F>
RIPP_HD Aff<F> pow2_mul(const Team& tm, const Aff<F>& p, int h) {
  Jac<F> a = Jac<F>::from_affine(p);
#pragma unroll 1
  for (int i = 0; i < h; i++) a = dbl<F>(tm, a);
  return to_affine<F>(tm, a);
}

// Same sum when every TEAM has its own scalar (element-wise scalings a_i r^i, ck_i r^-i of groth16_aggregation.rs:118-131,
// SIPP's a_i r_i): all teams of a warp walk the same (bit, digit) slots -- `m` digits, `nbits` bits, the warp's maxima --
// and a slot whose digit is zero adds the identity, so no team ever skips an exchange.
template <class F>
RIPP_HD Jac<F> endo_mul_sel(const Team& tm, const Aff<F>& p, const EndoBits& c, int m, int nbits, uint32_t* bases) {
  constexpr int AW = sizeof(Aff<F>) / 4;
  {
    Aff<F> b = p;
    for (int t = 0; t < m; t++) {
      if (tm.t == 0) aff_st<F>(bases + t * AW, b);
      if (t + 1 < m) b = endo_map(b);
    }
  }
  sync(tm);
  Jac<F> acc = Jac<F>::inf();
#pragma unroll 1
  for (int j = nbits - 1; j >= 0; j--) {
    acc = dbl<F>(tm, acc);
#pragma unroll 1
    for (int t = 0; t < m; t++) {
      const bool ps = (c.pos[t][j >> 5] >> (j & 31)) & 1, ng = (c.neg[t][j >> 5] >> (j & 31)) & 1;
      Aff<F> q = aff_ld<F>(bases + t * AW);
      if (ng) q = q.neg();
      if (!(ps || ng)) q = Aff<F>::inf();
      acc = madd<F>(tm, acc, q);
    }
  }
  return acc;
}

}  // namespace xt
}  // namespace ripp
