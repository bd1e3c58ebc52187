// Multi-Miller loop and final exponentiation on the six-lane Fq12 engine (l6.cuh).
// Replaces cfg_multi_pairing's hot loop (inner_products/src/lib.rs:83-115): one (G1, G2) pair per
// six-lane group, five groups per warp, the warp's five Miller values multiplied in shared memory,
// one Fq12 partial per warp, a tree of group products, and one group per final exponentiation.
#include "common.cuh"
#include "l6.cuh"

using namespace ripp::l6;

static __device__ __forceinline__ int tower_slot(int k) { return (k & 1) * 3 + (k >> 1); }

struct Miller6Batch {
  const G1Aff* p[RIPP_MAX_BATCH];
  const G2Aff* q[RIPP_MAX_BATCH];
  uint32_t n, wps;  // pairs per segment, warps per segment (5 * KP pairs per warp)
  int nseg;
  uint32_t fixed_q;  // PER_GROUP kernels: bit j set = pair j of every item has the one Q at q[j][0]
};
// TAB kernels (k_miller6<.., .., false, true>): any number of segments, segment s's P and Q base pointers at
// segs[2 s], segs[2 s + 1] in device memory (b.p[0] holds segs); b.nseg segments of b.n pairs
struct M6Seg {
  const G1Aff* p;
  const G2Aff* q;
};

constexpr int M6_NREG = 2;
constexpr int M6_WARPS = 4;
RIPP_HD constexpr int m6_smem_bytes(int kp) { return (M6_WARPS * 5 * group_words(M6_NREG, kp) + 16) * 4; }

// the generator of G2 in global memory: Q of masked pairs (identities / padding) -- per device, written by
// ripp_pairing6_init_device
__device__ G2Aff g_g2_gen;
__global__ void k_init_g2_gen() { g_g2_gen = g2_generator(); }

// KP pairs per six-lane group share one accumulator (one Fq12 squaring per bit instead of KP):
// KP = 1 minimises latency (late GIPA rounds), KP = 4 maximises throughput (long vectors).
// PER_GROUP: one Miller value per item instead of one product per warp -- group t walks pair j = (p[j][t], q[j][t]) for
// j < KP (one segment of n items; Q of pair j is q[j][0] for every item when bit j of fixed_q is set) and writes its
// accumulator to partials[t] (the per-proof values of a Groth16 batch, groth16.cu).
// TAB: the segments' base pointers come from the device table at b.p[0] (M6Seg), the segment from the flat warp index.
template <int WARPS, int KP, bool PER_GROUP = false, bool TAB = false>
__global__ void __launch_bounds__(32 * WARPS) k_miller6(Miller6Batch b, Fq12* __restrict__ partials) {
  extern __shared__ __align__(16) uint32_t smem[];
  constexpr int GW = group_words(M6_NREG, KP);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // five groups per warp; lanes 30, 31 MIRROR lanes 24, 25 (coefficients 0, 1 of group 4: same addresses, same values),
  // so no sixth scratch slot is needed: 18.4 KB of shared memory per warp at KP = 4.  (Three CTAs per SM then fit, but the
  // 168-register build that needs spills: Miller 2^16 19.5 -> 25.3 ms, measured; the room goes to more pairs per group.)
  const int g = lane < 30 ? lane / 6 : 4;
  uint32_t* wsm = smem + warp * 5 * GW;
  Ctx c{lane % 6, wsm + g * GW};
  c.zero = smem + WARPS * 5 * GW;  // l6.cuh's padding operand: sixteen words behind the groups, one slot per CTA
  if (threadIdx.x < 12) smem[WARPS * 5 * GW + threadIdx.x] = 0;
  __syncthreads();
  uint32_t* pairs = c.sm + OFF_F + M6_NREG * F12W;
  const uint32_t gw = blockIdx.x * WARPS + warp;
  const uint32_t seg = gw / b.wps, wl = gw % b.wps;
  // lane 0 of each group stages its pairs; identities / padding run on the generators and are masked
  if (c.k == 0) {
    for (int j = 0; j < KP; j++) {
      const uint32_t i = PER_GROUP ? wl * 5 + g : (wl * 5 + g) * KP + j;
      const int sv = PER_GROUP ? j : (int)seg;
      G1Aff P = g1_generator();
      const G2Aff* Q = &g_g2_gen;
      uint32_t valid = 0;
      if constexpr (TAB) {
        if (seg < (uint32_t)b.nseg && i < b.n) {
          const M6Seg sg = reinterpret_cast<const M6Seg*>(b.p[0])[seg];
          G1Aff p = sg.p[i];
          const G2Aff* q = &sg.q[i];
          if (!p.is_inf() && !q->is_inf()) {
            P = p;
            Q = q;
            valid = 1;
          }
        }
      } else if (seg < (uint32_t)b.nseg && i < b.n) {
        G1Aff p = b.p[sv][i];
        const G2Aff* q = &b.q[sv][PER_GROUP && ((b.fixed_q >> j) & 1) ? 0 : i];
        if (!p.is_inf() && !q->is_inf()) {
          P = p;
          Q = q;
          valid = 1;
        }
      }
      uint32_t* pb = pairs + j * PAIR_WORDS;
      stage_pair_p(pb, P);
      set_pair_q(pb, Q);
      pb[PB_VALID] = valid;
    }
  }
  __syncwarp();
  miller(c, pairs, KP);
  if constexpr (PER_GROUP) {
    const uint32_t t = wl * 5 + g;
    if (lane < 30 && seg < (uint32_t)b.nseg && t < b.n)
      reinterpret_cast<Fq2*>(&partials[t])[tower_slot(c.k)] = ld2(freg(c, 0) + c.k * FQ2W);
    return;
  }
  // product of the five groups' values: (0 <- 0*1, 2 <- 2*3), 0 <- 0*2, 0 <- 0*4; idle groups write their junk register
  uint32_t* F0 = freg(c, 0);
  uint32_t* J = freg(c, 1);
  auto other = [&](int gg) { return wsm + gg * GW + OFF_F; };
  mul_p(c, (g == 0 || g == 2) ? F0 : J, F0, other(g == 0 ? 1 : (g == 2 ? 3 : g)));
  mul_p(c, g == 0 ? F0 : J, F0, other(g == 0 ? 2 : g));
  mul_p(c, g == 0 ? F0 : J, F0, other(g == 0 ? 4 : g));
  if (g == 0 && seg < (uint32_t)b.nseg) {
    Fq2* out = reinterpret_cast<Fq2*>(&partials[gw]);
    out[tower_slot(c.k)] = ld2(F0 + c.k * FQ2W);
  }
}

// out[s][j] = prod in[s][j*R .. min(T, j*R+R)) ; one group per output, five groups per warp
constexpr int R6_GROUP_WORDS = group_words(2, 0);
template <int WARPS>
__global__ void __launch_bounds__(32 * WARPS) k_reduce6(const Fq12* __restrict__ in, uint32_t T, uint32_t R, uint32_t To,
                                                       Fq12* __restrict__ out, uint32_t total) {
  extern __shared__ __align__(16) uint32_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane / 6;
  Ctx c{lane % 6, smem + (warp * 6 + g) * R6_GROUP_WORDS};
  uint32_t t = (blockIdx.x * WARPS + warp) * 5 + g;
  bool live = g < 5 && t < total;
  uint32_t s = live ? t / To : 0, j = live ? t % To : 0;
  uint32_t lo = j * R, hi = lo + R < T ? lo + R : T;
  const Fq2* src = reinterpret_cast<const Fq2*>(in + (size_t)s * T);
  st2(freg(c, 0) + c.k * FQ2W, src[(size_t)lo * 6 + tower_slot(c.k)]);
  __syncwarp();
  for (uint32_t r = 1; r < R; r++) {  // uniform trip count; rows past `hi` multiply by one
    bool on = lo + r < hi;
    Fq2 v = on ? src[(size_t)(lo + r) * 6 + tower_slot(c.k)] : f2sel(c.k == 0, Fq2::one(), Fq2::zero());
    st2(freg(c, 1) + c.k * FQ2W, v);
    __syncwarp();
    mul(c, 0, 0, 1);
  }
  if (live) reinterpret_cast<Fq2*>(out + t)[tower_slot(c.k)] = ld2(freg(c, 0) + c.k * FQ2W);
}

// out[s] = final_exponentiation(prod_j in[s][j]), j < T (T <= 8); one group per value
constexpr int FE_NREG = 9;
constexpr int FE_GROUP_WORDS = group_words(FE_NREG, 0);
__global__ void __launch_bounds__(64) k_final_exp6(const Fq12* __restrict__ in, uint32_t T, Fq12* __restrict__ out, int nseg) {
  extern __shared__ __align__(16) uint32_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane / 6;
  Ctx c{lane % 6, smem + (warp * 6 + g) * FE_GROUP_WORDS};
  int s = (blockIdx.x * 2 + warp) * 5 + g;
  bool live = g < 5 && s < nseg;
  const Fq2* src = reinterpret_cast<const Fq2*>(in + (size_t)(live ? s : 0) * T);
  st2(freg(c, 0) + c.k * FQ2W, src[tower_slot(c.k)]);
  __syncwarp();
  for (uint32_t r = 1; r < T; r++) {
    st2(freg(c, 8) + c.k * FQ2W, src[(size_t)r * 6 + tower_slot(c.k)]);
    __syncwarp();
    mul(c, 0, 0, 8);
  }
  final_exp(c);
  if (live) reinterpret_cast<Fq2*>(out + s)[tower_slot(c.k)] = ld2(freg(c, 0) + c.k * FQ2W);
}


// The Groth16 check of one proof per group: final_exponentiation(in[t]) == e(alpha, beta) (`ab`, 576 B), compared on
// canonical Fq values (from_mont of any 384-bit value is the fully reduced product).  out[t] = 1 / 0, or with `pre`
// (decode statuses of the serialized entry) pre[t] when non-zero, else RIPP_GROTH16_OK / RIPP_GROTH16_REJECTED.
// ab_stride 1: one target per item, ab[t] (the pairing equations of the aggregate verifier, ripp_pairing_checks_l6).
__global__ void __launch_bounds__(64) k_groth16_check6(const Fq12* __restrict__ in, const Fq12* __restrict__ ab, uint32_t ab_stride,
                                                       uint32_t n, const uint8_t* pre, uint8_t* out) {  // pre may alias out
  extern __shared__ __align__(16) uint32_t smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = lane / 6;
  Ctx c{lane % 6, smem + (warp * 6 + g) * FE_GROUP_WORDS};
  const uint32_t t = (blockIdx.x * 2 + warp) * 5 + g;
  const bool live = g < 5 && t < n;
  st2(freg(c, 0) + c.k * FQ2W, reinterpret_cast<const Fq2*>(in + (live ? t : 0))[tower_slot(c.k)]);
  __syncwarp();
  final_exp(c);
  const Fq2 f = ld2(freg(c, 0) + c.k * FQ2W), e = reinterpret_cast<const Fq2*>(ab + (live ? t : 0) * ab_stride)[tower_slot(c.k)];
  const bool eq = f.c0.from_mont() == e.c0.from_mont() && f.c1.from_mont() == e.c1.from_mont();
  const uint32_t all = __ballot_sync(0xffffffffu, eq);
  if (live && c.k == 0) {
    const bool ok = ((all >> (6 * g)) & 0x3fu) == 0x3fu;
    out[t] = pre ? (pre[t] ? pre[t] : (ok ? RIPP_GROTH16_OK : RIPP_GROTH16_REJECTED)) : (uint8_t)ok;
  }
}

// out[i] = in[i]^sc[i] (GT exponentiation by an Fr scalar in Montgomery form); one group per element.
// The verifiers' `mul_helper` on PairingOutput (ip_proofs/src/lib.rs:15-19 with T = GT; gipa.rs:355-357,
// sipp/src/lib.rs:148-156).
constexpr int GP_NREG = 5;
constexpr int GP_GROUP_WORDS = group_words(GP_NREG, 0);
__global__ void __launch_bounds__(32) k_gt_pow6(const Fq12* __restrict__ in, const Fr* __restrict__ sc, uint32_t n,
                                                Fq12* __restrict__ out) {
  extern __shared__ __align__(16) uint32_t smem[];
  const int lane = threadIdx.x & 31;
  const int g = lane / 6;
  Ctx c{lane % 6, smem + g * GP_GROUP_WORDS};
  uint32_t t = blockIdx.x * 5 + g;
  bool live = g < 5 && t < n;
  const Fq2* src = reinterpret_cast<const Fq2*>(in + (live ? t : 0));
  st2(freg(c, 1) + c.k * FQ2W, src[tower_slot(c.k)]);
  uint32_t* e = c.sm + OFF_LINE;  // the line slot is free here: holds the canonical exponent
  if (c.k == 0) {
    Fr s = live ? sc[t].from_mont() : Fr::zero();
    for (int i = 0; i < 8; i++) e[i] = s.v[i];
  }
  __syncwarp();
  pow_fr(c, 0, 1, 2, 3, 4, e);
  if (live) reinterpret_cast<Fq2*>(out + t)[tower_slot(c.k)] = ld2(freg(c, 0) + c.k * FQ2W);
}

// ------------------------------------------------------------------------------------------------
// W = 3 shape (l6.cuh): ONE Fq12 per warp on 18 lanes.  For the latency-bound end of the path -- the late GIPA
// rounds, every final exponentiation, the verifiers' GT powers -- where there are fewer Fq12 chains than
// sub-partitions and the length of ONE chain is the whole cost.
// ------------------------------------------------------------------------------------------------
static __device__ __forceinline__ Ctx3 ctx18(uint32_t* wsm, int group_words_no_bus) {
  const int vl = (threadIdx.x & 31) % 18;  // lanes 18..31 mirror lanes 0..13: same addresses, same values
  if ((threadIdx.x & 31) < 12) wsm[group_words_no_bus + BUS_ZERO + (threadIdx.x & 31)] = 0;  // l6.cuh's padding operand
  __syncwarp();
  return Ctx3{vl / 3, wsm, nullptr, vl % 3, wsm + group_words_no_bus, 0, wsm + group_words_no_bus + BUS_ZERO};
}
constexpr int M18_WARPS = 4;
constexpr int M18_GROUP_WORDS = group_words(M6_NREG, 1) + BUS_TOTAL;

// grid (ceil(n / 4), nseg): warp w of segment s walks pair w; the CTA's four Miller values are multiplied in shared
// memory; one partial per CTA at partials[s * gridDim.x + blockIdx.x].
__global__ void __launch_bounds__(32 * M18_WARPS) k_miller18(Miller6Batch b, Fq12* __restrict__ partials) {
  extern __shared__ __align__(16) uint32_t smem[];
  const int warp = threadIdx.x >> 5;
  uint32_t* wsm = smem + warp * M18_GROUP_WORDS;
  Ctx3 c = ctx18(wsm, group_words(M6_NREG, 1));
  uint32_t* pairs = c.sm + OFF_F + M6_NREG * F12W;
  const uint32_t seg = blockIdx.y, i = blockIdx.x * M18_WARPS + warp;
  if (c.k == 0 && c.role == 0) {
    G1Aff P = g1_generator();
    const G2Aff* Q = &g_g2_gen;
    uint32_t valid = 0;
    if (i < b.n) {
      G1Aff p = b.p[seg][i];
      const G2Aff* q = &b.q[seg][i];
      if (!p.is_inf() && !q->is_inf()) {
        P = p;
        Q = q;
        valid = 1;
      }
    }
    stage_pair_p(pairs, P);
    set_pair_q(pairs, Q);
    pairs[PB_VALID] = valid;
  }
  __syncwarp();
  miller(c, pairs, 1);
  uint32_t* F0 = freg(c, 0);
  auto other = [&](int w) { return smem + w * M18_GROUP_WORDS + OFF_F; };
  __syncthreads();
  if ((warp & 1) == 0) mul_p(c, F0, F0, other(warp + 1));
  __syncthreads();
  if (warp == 0) {
    mul_p(c, F0, F0, other(2));
    if (c.role == 0) {
      Fq2* out = reinterpret_cast<Fq2*>(&partials[(size_t)seg * gridDim.x + blockIdx.x]);
      out[tower_slot(c.k)] = ld2(F0 + c.k * FQ2W);
    }
  }
}

// out[s][j] = prod in[s][j*R .. min(T, j*R+R)); one warp per output
constexpr int R18_GROUP_WORDS = group_words(2, 0) + BUS_TOTAL;
__global__ void __launch_bounds__(32 * M18_WARPS) k_reduce18(const Fq12* __restrict__ in, uint32_t T, uint32_t R, uint32_t To,
                                                            Fq12* __restrict__ out, uint32_t total) {
  extern __shared__ __align__(16) uint32_t smem[];
  const int warp = threadIdx.x >> 5;
  Ctx3 c = ctx18(smem + warp * R18_GROUP_WORDS, group_words(2, 0));
  uint32_t t = blockIdx.x * M18_WARPS + warp;
  bool live = t < total;
  uint32_t s = live ? t / To : 0, j = live ? t % To : 0;
  uint32_t lo = j * R, hi = lo + R < T ? lo + R : T;
  const Fq2* src = reinterpret_cast<const Fq2*>(in + (size_t)s * T);
  st2(freg(c, 0) + c.k * FQ2W, src[(size_t)lo * 6 + tower_slot(c.k)]);
  __syncwarp();
  for (uint32_t r = 1; r < R; r++) {
    bool on = lo + r < hi;
    Fq2 v = on ? src[(size_t)(lo + r) * 6 + tower_slot(c.k)] : f2sel(c.k == 0, Fq2::one(), Fq2::zero());
    st2(freg(c, 1) + c.k * FQ2W, v);
    __syncwarp();
    mul(c, 0, 0, 1);
  }
  if (live && c.role == 0) reinterpret_cast<Fq2*>(out + t)[tower_slot(c.k)] = ld2(freg(c, 0) + c.k * FQ2W);
}

// out[s] = final_exponentiation(prod_j in[s][j]), j < T; one warp (one CTA) per value
constexpr int FE18_GROUP_WORDS = group_words(FE_NREG, 0) + BUS_TOTAL;
__global__ void __launch_bounds__(32) k_final_exp18(const Fq12* __restrict__ in, uint32_t T, Fq12* __restrict__ out) {
  extern __shared__ __align__(16) uint32_t smem[];
  Ctx3 c = ctx18(smem, group_words(FE_NREG, 0));
  const int s = blockIdx.x;
  const Fq2* src = reinterpret_cast<const Fq2*>(in + (size_t)s * T);
  st2(freg(c, 0) + c.k * FQ2W, src[tower_slot(c.k)]);
  __syncwarp();
  for (uint32_t r = 1; r < T; r++) {
    st2(freg(c, 8) + c.k * FQ2W, src[(size_t)r * 6 + tower_slot(c.k)]);
    __syncwarp();
    mul(c, 0, 0, 8);
  }
  final_exp(c);
  if (c.role == 0) reinterpret_cast<Fq2*>(out + s)[tower_slot(c.k)] = ld2(freg(c, 0) + c.k * FQ2W);
}

// out[i] = in[i]^sc[i], one warp per element (k_gt_pow6 on eighteen lanes)
constexpr int GP18_GROUP_WORDS = group_words(GP_NREG, 0) + BUS_TOTAL;
__global__ void __launch_bounds__(32) k_gt_pow18(const Fq12* __restrict__ in, const Fr* __restrict__ sc, uint32_t n,
                                                 Fq12* __restrict__ out) {
  extern __shared__ __align__(16) uint32_t smem[];
  Ctx3 c = ctx18(smem, group_words(GP_NREG, 0));
  const uint32_t t = blockIdx.x;
  const Fq2* src = reinterpret_cast<const Fq2*>(in + t);
  st2(freg(c, 1) + c.k * FQ2W, src[tower_slot(c.k)]);
  uint32_t* e = c.sm + OFF_LINE;  // the line slot is free here: holds the canonical exponent
  if (c.k == 0 && c.role == 0) {
    Fr s = sc[t].from_mont();
    for (int i = 0; i < 8; i++) e[i] = s.v[i];
  }
  __syncwarp();
  pow_fr(c, 0, 1, 2, 3, 4, e);
  if (c.role == 0) reinterpret_cast<Fq2*>(out + t)[tower_slot(c.k)] = ld2(freg(c, 0) + c.k * FQ2W);
}

// number of warps the eighteen-lane kernels may occupy before the throughput shape takes over: two per
// sub-partition (a third warp on a sub-partition queues behind the same multiplier pipe).  RIPP_B200_L18_WARPS overrides.
static size_t l18_max_warps() {
  static const long v = [] {
    const char* e = getenv("RIPP_B200_L18_WARPS");
    return e ? atol(e) : 1184L;
  }();
  return (size_t)v;
}

// GT membership of untrusted Fq12 values (what ark-serialize's Valid::check establishes for PairingOutput when the
// reference deserialises a proof): f is in the cyclotomic subgroup, f^(p^4) f == f^(p^2), and f^p == f^x
// (Scott, ePrint 2021/1130; oracle: gt_in_subgroup_fast, checked there against f^r == 1).  One group per element;
// a failing element ORs `flag` into bad[0], or into bad[owner[i]] when owner is given (one word per aggregate).
constexpr int GC_NREG = 3;
constexpr int GC_GROUP_WORDS = group_words(GC_NREG, 0) + BUS_TOTAL;
__global__ void __launch_bounds__(32) k_gt_check18(const Fq12* __restrict__ in, uint32_t n, uint32_t* __restrict__ bad,
                                                   uint32_t flag, const uint32_t* __restrict__ owner) {
  extern __shared__ __align__(16) uint32_t smem[];
  Ctx3 c = ctx18(smem, group_words(GC_NREG, 0));
  const Fq2* src = reinterpret_cast<const Fq2*>(in + blockIdx.x);
  st2(freg(c, 0) + c.k * FQ2W, src[tower_slot(c.k)]);
  __syncwarp();
  frob(c, 1, 0, 2);
  frob(c, 2, 1, 2);
  mul(c, 2, 2, 0);
  bool ne = !(ld2(freg(c, 2) + c.k * FQ2W) == ld2(freg(c, 1) + c.k * FQ2W));
  __syncwarp();
  exp_by_x(c, 2, 0);  // cyclotomic squarings: meaningful only when the first test passed, and only then consulted
  frob(c, 1, 0, 1);
  ne = ne || !(ld2(freg(c, 2) + c.k * FQ2W) == ld2(freg(c, 1) + c.k * FQ2W));
  if (ne) atomicOr(bad + (owner ? owner[blockIdx.x] : 0), flag);
}
int ripp_gt_check_l6(ripp_ctx* ctx, const void* in, size_t n, uint32_t* bad_dev, uint32_t flag, const uint32_t* owner_dev) {
  if (n == 0) return RIPP_OK;
  k_gt_check18<<<(unsigned)n, 32, GC_GROUP_WORDS * 4, ctx->stream>>>((const Fq12*)in, (uint32_t)n, bad_dev, flag, owner_dev);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// k_reduce6 levels over nseg runs of *T partials each, run s at *src + s * *T: out[s][j] = prod in[s][j*R .. j*R+R), R = 8,
// until at most `stop` are left per run.  The level that leaves one per run writes to `last` when given, else the levels
// ping-pong between *src and dst.  *src and *T then hold the result.
static int reduce6(ripp_ctx* ctx, uint32_t nseg, uint32_t stop, Fq12** src, Fq12* dst, uint32_t* T, Fq12* last = nullptr) {
  const uint32_t R = 8;
  while (*T > stop) {
    const uint32_t To = (*T + R - 1) / R, tot = nseg * To;
    Fq12* o = To == 1 && last ? last : dst;
    k_reduce6<M6_WARPS><<<(tot + 5 * M6_WARPS - 1) / (5 * M6_WARPS), 32 * M6_WARPS, M6_WARPS * 6 * R6_GROUP_WORDS * 4, ctx->stream>>>(
        *src, *T, R, To, o, tot);
    LAUNCHED(ctx);
    dst = *src;
    *src = o;
    *T = To;
  }
  return RIPP_OK;
}

// out[s] = prod_i in[s * n + i]^sc[s * n + i], s < nseg  (device memory; in: nseg x n Fq12, sc: nseg x n Fr Montgomery)
int ripp_gt_multiexp_l6(ripp_ctx* ctx, const void* in, const void* sc, size_t n, void* out, int nseg) {
  CU(cudaSetDevice(ctx->device));
  if (n == 0) {
    Fq12 one = Fq12::one();
    CU(cudaMemcpyAsync(out, &one, sizeof(one), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return RIPP_OK;
  }
  const size_t total = (size_t)nseg * n;
  void *bufA, *bufB;
  OK(scratch(ctx, 17, total * sizeof(Fq12) + 4096, &bufA));
  OK(scratch(ctx, 18, total * sizeof(Fq12) / 4 + 8192, &bufB));
  TimeScope ts_(ctx, RIPP_T_OTHER);
  if (total <= l18_max_warps())
    k_gt_pow18<<<(unsigned)total, 32, GP18_GROUP_WORDS * 4, ctx->stream>>>((const Fq12*)in, (const Fr*)sc, (uint32_t)total,
                                                                         n == 1 ? (Fq12*)out : (Fq12*)bufA);
  else
    k_gt_pow6<<<(unsigned)((total + 4) / 5), 32, 6 * GP_GROUP_WORDS * 4, ctx->stream>>>((const Fq12*)in, (const Fr*)sc,
                                                                                        (uint32_t)total, n == 1 ? (Fq12*)out : (Fq12*)bufA);
  LAUNCHED(ctx);
  Fq12* src = (Fq12*)bufA;
  uint32_t T = (uint32_t)n;
  return reduce6(ctx, (uint32_t)nseg, 1, &src, (Fq12*)bufB, &T, (Fq12*)out);
}

// Pairs per six-lane group for nseg segments of pairs_per_seg pairs (the pairs of a group share the accumulator's
// squaring).  All warps of a launch do equal work, so the launch takes ceil(warps / resident warps) waves of one warp's
// duration; per doubling step a warp spends ~2040 MAC32 on the shared squaring and ~3096 per pair (point step + sparse
// line product).  Pick the kp in {1..4} with the cheapest waves x duration -- e.g. 12 288 pairs (TIPP 2^12, first
// round): kp = 2 is two waves, kp = 3 one.  RIPP_B200_M6_KP pins kp; background work takes 4.  `many_waves`: a launch of
// three or more waves at kp = 4 takes kp = 4 without the comparison.  The RLC check passes false: at n = 100 000
// (1725 segments) that shortcut's kp = 4 measured 56.3 ms against 55.6 ms at the compared kp = 3 (DESIGN.md §6).
static int m6_pairs_per_group(ripp_ctx* ctx, size_t nseg, size_t pairs_per_seg, bool many_waves, int* kp_out) {
  int sms = 0;
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ctx->device));
  const size_t resident = (size_t)sms * 2 * M6_WARPS;  // two CTAs per SM (255 registers)
  int kp = 4;
  double best = 0;
  // many waves: CTAs are scheduled as others retire, the tail of the last wave is a small share -- most sharing wins
  // (six or eight pairs per group fit the shared memory since Q left the pair block, but measured no better: 2^18 pairs
  // 77.3 ms at kp = 4, 80.2 at 6, 78.9 at 8; 2^16: 19.7 / 19.4 / 23.8 ms)
  const bool many = many_waves && nseg * ((pairs_per_seg + 19) / 20) >= 3 * resident;
  for (int k = 1; k <= 4 && !many; k++) {
    const size_t warps = nseg * ((pairs_per_seg + 5 * k - 1) / (5 * k));
    const double t = (double)((warps + resident - 1) / resident) * (2040.0 + 3096.0 * k);
    if (k == 1 || t <= best) {
      best = t;
      kp = k;
    }
  }
  static const int force = [] {
    const char* e = getenv("RIPP_B200_M6_KP");
    return e ? atoi(e) : 0;
  }();
  if (force >= 1 && force <= 4) kp = force;
  if (ctx->background) kp = 4;
  *kp_out = kp;
  return RIPP_OK;
}

template <int KP, bool TAB = false>
static int launch_miller6(ripp_ctx* ctx, Miller6Batch& b, Fq12* dst) {
  b.wps = (uint32_t)(((size_t)b.n + 5 * KP - 1) / (5 * KP));
  const size_t nwarps = (size_t)b.wps * b.nseg;
  k_miller6<M6_WARPS, KP, false, TAB><<<(unsigned)((nwarps + M6_WARPS - 1) / M6_WARPS), 32 * M6_WARPS, m6_smem_bytes(KP), ctx->stream>>>(
      b, dst);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// The six-lane products: one k_miller6 launch at kp pairs per group (one partial per warp, at *src), then reduce6 over
// nseg equal runs of those partials down to `stop` per run.  The runs are b's segments, or (the RLC check) the
// warp-aligned segments inside b's one segment.
template <bool TAB = false>
static int m6_products(ripp_ctx* ctx, Miller6Batch& b, int kp, uint32_t nseg, uint32_t stop, Fq12** src, Fq12* dst, uint32_t* T) {
  if (kp == 4)
    OK((launch_miller6<4, TAB>(ctx, b, *src)));
  else if (kp == 3)
    OK((launch_miller6<3, TAB>(ctx, b, *src)));
  else if (kp == 2)
    OK((launch_miller6<2, TAB>(ctx, b, *src)));
  else
    OK((launch_miller6<1, TAB>(ctx, b, *src)));
  *T = (uint32_t)((size_t)b.wps * b.nseg / nseg);
  return reduce6(ctx, nseg, stop, src, dst, T);
}

int ripp_pairing_batch_l6(ripp_ctx* ctx, int nseg, const void* const* g1, const void* const* g2, size_t n, void* out,
                          bool with_final_exp) {
  if (nseg <= 0 || nseg > RIPP_MAX_BATCH) return fail(RIPP_ERR_ARG, "bad segment count");
  CU(cudaSetDevice(ctx->device));
  Fq12 one = Fq12::one();
  if (n == 0) {
    for (int s = 0; s < nseg; s++)
      CU(cudaMemcpyAsync((char*)out + 576 * s, &one, sizeof(one), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    return RIPP_OK;
  }
  Miller6Batch b;
  b.nseg = nseg;
  b.n = (uint32_t)n;
  for (int s = 0; s < nseg; s++) {
    b.p[s] = (const G1Aff*)g1[s];
    b.q[s] = (const G2Aff*)g2[s];
  }
  size_t total = (size_t)nseg * n;
  size_t max_partials = (size_t)nseg * ((n + 3) / 4 + 1);
  void *bufA, *bufB;
  OK(scratch(ctx, 2, max_partials * sizeof(Fq12) + 4096, &bufA));
  OK(scratch(ctx, 3, max_partials * sizeof(Fq12) / 4 + 8192, &bufB));
  Fq12 *src = (Fq12*)bufA, *dst = (Fq12*)bufB;
  uint32_t T;
  if (total <= l18_max_warps()) {
    // latency shape: one pair per eighteen-lane warp, up to l18_max_warps pairs (two warps per sub-partition); four
    // warps per CTA combined in shared memory, then a tree of one-warp products and one warp per final exponentiation.
    // Above that the six-lane shape wins, also against two or four pairs per eighteen-lane warp -- measured: six products
    // of 256 / 512 pairs 3.80 / 5.68 ms with 2 / 4 pairs per eighteen-lane warp, 3.18 / 3.69 ms on six lanes; TIPP 2^12
    // 93.5 -> 87.8 ms.
    TimeScope ts_(ctx, RIPP_T_MILLER);
    const uint32_t ctas = ((uint32_t)n + M18_WARPS - 1) / M18_WARPS;
    k_miller18<<<dim3(ctas, nseg), 32 * M18_WARPS, M18_WARPS * M18_GROUP_WORDS * 4, ctx->stream>>>(b, src);
    LAUNCHED(ctx);
    T = ctas;
    const uint32_t R = 4, stop = with_final_exp ? R : 1;
    while (T > stop) {
      uint32_t To = (T + R - 1) / R, tot = (uint32_t)nseg * To;
      k_reduce18<<<(tot + M18_WARPS - 1) / M18_WARPS, 32 * M18_WARPS, M18_WARPS * R18_GROUP_WORDS * 4, ctx->stream>>>(src, T, R, To,
                                                                                                                   dst, tot);
      LAUNCHED(ctx);
      Fq12* t = src;
      src = dst;
      dst = t;
      T = To;
    }
  } else {
    // throughput shape: several pairs per six-lane group, the k_reduce6 tree down to at most four partials per segment
    // for k_final_exp18 (one without it)
    int kp;
    OK(m6_pairs_per_group(ctx, nseg, n, true, &kp));
    TimeScope ts_(ctx, RIPP_T_MILLER);
    OK(m6_products(ctx, b, kp, nseg, with_final_exp ? 4 : 1, &src, dst, &T));
  }
  if (!with_final_exp) {
    CU(cudaMemcpyAsync(out, src, (size_t)nseg * sizeof(Fq12), cudaMemcpyDeviceToDevice, ctx->stream));
    return RIPP_OK;
  }
  TimeScope ts2_(ctx, RIPP_T_FINAL_EXP);
  k_final_exp18<<<nseg, 32, FE18_GROUP_WORDS * 4, ctx->stream>>>(src, T, (Fq12*)out);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// nseg products of n pairs with the segments' pointers in device memory (M6Seg table, any nseg): one k_miller6<.., TAB>
// launch at the pairs-per-group rule's kp, the k_reduce6 tree down to at most four partials per segment, one final
// exponentiation launch.  The launch count depends on n and kp, not on nseg beyond the kp choice.  Scratch slots
// slot0, slot0 + 1.
int ripp_pairing_table_l6(ripp_ctx* ctx, const void* segs_dev, size_t nseg, size_t n, void* out, int slot0) {
  if (nseg == 0) return RIPP_OK;
  if (n == 0 || nseg > 0xffffffffu / ((n + 4) / 5)) return fail(RIPP_ERR_ARG, "bad pairing table shape");
  CU(cudaSetDevice(ctx->device));
  Miller6Batch b;
  memset(&b, 0, sizeof(b));
  b.p[0] = (const G1Aff*)segs_dev;
  b.n = (uint32_t)n;
  b.nseg = (int)nseg;
  int kp;
  OK(m6_pairs_per_group(ctx, nseg, n, true, &kp));
  const size_t max_partials = nseg * ((n + 4) / 5);
  void *bufA, *bufB;
  OK(scratch(ctx, slot0, max_partials * sizeof(Fq12) + 4096, &bufA));
  OK(scratch(ctx, slot0 + 1, nseg * (((n + 4) / 5 + 7) / 8) * sizeof(Fq12) + 8192, &bufB));  // the first k_reduce6 level
  Fq12 *src = (Fq12*)bufA, *dst = (Fq12*)bufB;
  uint32_t T;
  {
    TimeScope ts_(ctx, RIPP_T_MILLER);
    OK(m6_products<true>(ctx, b, kp, (uint32_t)nseg, 4, &src, dst, &T));
  }
  return ripp_final_exp_l6(ctx, src, T, out, (int)nseg);
}

// out[s] = final_exponentiation(prod_j in[s*T + j])
int ripp_final_exp_l6(ripp_ctx* ctx, const void* in, uint32_t T, void* out, int nseg) {
  CU(cudaSetDevice(ctx->device));
  TimeScope ts_(ctx, RIPP_T_FINAL_EXP);
  if ((size_t)nseg <= l18_max_warps())
    k_final_exp18<<<nseg, 32, FE18_GROUP_WORDS * 4, ctx->stream>>>((const Fq12*)in, T, (Fq12*)out);
  else
    k_final_exp6<<<(nseg + 9) / 10, 64, 2 * 6 * FE_GROUP_WORDS * 4, ctx->stream>>>((const Fq12*)in, T, (Fq12*)out, nseg);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// Groth16 verification of n proofs, one six-lane group per proof (groth16.cu): the three pairs (A, B), (P, -gamma),
// (C, -delta) of a proof share one accumulator (KP = 3), then one final exponentiation and the compare per group.
// `miller` holds n Fq12.
int ripp_groth16_pairings_l6(ripp_ctx* ctx, const void* a, const void* b, const void* p, const void* c, const void* neg_gamma,
                             const void* neg_delta, const void* ab, size_t n, void* miller, const uint8_t* pre, uint8_t* out) {
  Miller6Batch mb;
  memset(&mb, 0, sizeof(mb));
  mb.p[0] = (const G1Aff*)a;
  mb.q[0] = (const G2Aff*)b;
  mb.p[1] = (const G1Aff*)p;
  mb.q[1] = (const G2Aff*)neg_gamma;
  mb.p[2] = (const G1Aff*)c;
  mb.q[2] = (const G2Aff*)neg_delta;
  mb.fixed_q = 0x6;
  mb.n = (uint32_t)n;
  mb.nseg = 1;
  mb.wps = (uint32_t)((n + 4) / 5);
  {
    TimeScope ts_(ctx, RIPP_T_MILLER);
    k_miller6<M6_WARPS, 3, true><<<(mb.wps + M6_WARPS - 1) / M6_WARPS, 32 * M6_WARPS, m6_smem_bytes(3), ctx->stream>>>(mb, (Fq12*)miller);
    LAUNCHED(ctx);
  }
  TimeScope ts_(ctx, RIPP_T_FINAL_EXP);
  k_groth16_check6<<<(unsigned)((n + 9) / 10), 64, 2 * 6 * FE_GROUP_WORDS * 4, ctx->stream>>>((const Fq12*)miller, (const Fq12*)ab, 0,
                                                                                            (uint32_t)n, pre, out);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// n pairing equations prod_{j < 3} e(p[j * n + t], q[j * n + t]) == tgt[t], one six-lane group per equation (the three
// pairs share one accumulator; a pair with an identity is left out); ok[t] = 1 / 0.  `miller` holds n Fq12.
int ripp_pairing_checks_l6(ripp_ctx* ctx, const void* p, const void* q, size_t n, void* miller, const void* tgt, uint8_t* ok) {
  Miller6Batch mb;
  memset(&mb, 0, sizeof(mb));
  for (int j = 0; j < 3; j++) {
    mb.p[j] = (const G1Aff*)p + j * n;
    mb.q[j] = (const G2Aff*)q + j * n;
  }
  mb.n = (uint32_t)n;
  mb.nseg = 1;
  mb.wps = (uint32_t)((n + 4) / 5);
  {
    TimeScope ts_(ctx, RIPP_T_MILLER);
    k_miller6<M6_WARPS, 3, true><<<(mb.wps + M6_WARPS - 1) / M6_WARPS, 32 * M6_WARPS, m6_smem_bytes(3), ctx->stream>>>(mb, (Fq12*)miller);
    LAUNCHED(ctx);
  }
  TimeScope ts_(ctx, RIPP_T_FINAL_EXP);
  k_groth16_check6<<<(unsigned)((n + 9) / 10), 64, 2 * 6 * FE_GROUP_WORDS * 4, ctx->stream>>>((const Fq12*)miller, (const Fq12*)tgt, 1,
                                                                                            (uint32_t)n, nullptr, ok);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// Pairs of the random-linear-combination check (groth16.cu verify_rlc): segment t of s proofs becomes sp pairs,
// (r_i A_i, B_i) for its proofs, then (P_t, -gamma), (C_t, -delta), then masked padding up to sp, a multiple of the
// pairs per warp, so that no warp's partial product straddles two segments.
__global__ void __launch_bounds__(64) k_rlc_pairs(const G1Aff* __restrict__ ra, const G2Aff* __restrict__ b,
                                                  const G1Aff* __restrict__ ps, const G1Aff* __restrict__ cs,
                                                  const G2Aff* __restrict__ neg_gamma, const G2Aff* __restrict__ neg_delta,
                                                  uint32_t n, uint32_t s, uint32_t sp, uint32_t nseg, G1Aff* __restrict__ P,
                                                  G2Aff* __restrict__ Q) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)nseg * sp) return;
  const uint32_t seg = (uint32_t)(t / sp), i = (uint32_t)(t % sp), lo = seg * s, len = min(s, n - lo);
  if (i < len) {
    P[t] = ra[lo + i];
    Q[t] = b[lo + i];
  } else if (i == len) {
    P[t] = ps[seg];
    Q[t] = *neg_gamma;
  } else {
    P[t] = i == len + 1 ? cs[seg] : G1Aff::inf();
    Q[t] = *neg_delta;
  }
}

int ripp_groth16_rlc_pairings_l6(ripp_ctx* ctx, const void* ra, const void* b, const void* ps, const void* cs, const void* neg_gamma,
                                 const void* neg_delta, const void* ab, size_t n, size_t s, size_t nseg, uint8_t* ok) {
  int kp;
  OK(m6_pairs_per_group(ctx, nseg, s + 2, false, &kp));  // a segment's s proofs and two fixed-Q pairs, before padding
  const size_t ppw = 5 * (size_t)kp, sp = (s + 2 + ppw - 1) / ppw * ppw, np = nseg * sp, T0 = sp / ppw;
  void *pq, *part;
  const size_t o_q = (np * sizeof(G1Aff) + 255) & ~(size_t)255;
  OK(scratch(ctx, 36, o_q + np * sizeof(G2Aff), &pq));
  const size_t o_b = (nseg * T0 * sizeof(Fq12) + 255) & ~(size_t)255;
  OK(scratch(ctx, 37, o_b + (nseg * ((T0 + 7) / 8) + 1) * sizeof(Fq12), &part));
  G1Aff* P = (G1Aff*)pq;
  G2Aff* Q = (G2Aff*)((char*)pq + o_q);
  Fq12 *src = (Fq12*)part, *dst = (Fq12*)((char*)part + o_b);
  {
    TimeScope ts_(ctx, RIPP_T_MILLER);
    k_rlc_pairs<<<(unsigned)((np + 63) / 64), 64, 0, ctx->stream>>>((const G1Aff*)ra, (const G2Aff*)b, (const G1Aff*)ps,
                                                                   (const G1Aff*)cs, (const G2Aff*)neg_gamma, (const G2Aff*)neg_delta,
                                                                   (uint32_t)n, (uint32_t)s, (uint32_t)sp, (uint32_t)nseg, P, Q);
    LAUNCHED(ctx);
    Miller6Batch mb;
    memset(&mb, 0, sizeof(mb));
    mb.p[0] = P;
    mb.q[0] = Q;
    mb.n = (uint32_t)np;
    mb.nseg = 1;
    // partials [seg * T0 + w] -> one Miller value per segment
    uint32_t T;
    OK(m6_products(ctx, mb, kp, (uint32_t)nseg, 1, &src, dst, &T));
  }
  TimeScope ts_(ctx, RIPP_T_FINAL_EXP);
  k_groth16_check6<<<(unsigned)((nseg + 9) / 10), 64, 2 * 6 * FE_GROUP_WORDS * 4, ctx->stream>>>(src, (const Fq12*)ab, 0, (uint32_t)nseg,
                                                                                               nullptr, ok);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// Opt-in shared-memory sizes of the six-lane kernels: function attributes are per device, set once per context
// creation (ripp_ctx_create) -- never from the launch paths, which run concurrently on several host threads.
int ripp_pairing6_init_device() {
  k_init_g2_gen<<<1, 1>>>();
  CU(cudaGetLastError());
  CU(cudaFuncSetAttribute(k_reduce6<M6_WARPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, M6_WARPS * 6 * R6_GROUP_WORDS * 4));
  CU(cudaFuncSetAttribute(k_final_exp6, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 6 * FE_GROUP_WORDS * 4));
  CU(cudaFuncSetAttribute(k_miller6<M6_WARPS, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, m6_smem_bytes(1)));
  CU(cudaFuncSetAttribute(k_miller6<M6_WARPS, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, m6_smem_bytes(2)));
  CU(cudaFuncSetAttribute(k_miller6<M6_WARPS, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, m6_smem_bytes(3)));
  CU(cudaFuncSetAttribute(k_miller6<M6_WARPS, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, m6_smem_bytes(4)));
  CU(cudaFuncSetAttribute(k_miller6<M6_WARPS, 3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, m6_smem_bytes(3)));
  CU(cudaFuncSetAttribute(k_miller6<M6_WARPS, 1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, m6_smem_bytes(1)));
  CU(cudaFuncSetAttribute(k_miller6<M6_WARPS, 2, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, m6_smem_bytes(2)));
  CU(cudaFuncSetAttribute(k_miller6<M6_WARPS, 3, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, m6_smem_bytes(3)));
  CU(cudaFuncSetAttribute(k_miller6<M6_WARPS, 4, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, m6_smem_bytes(4)));
  CU(cudaFuncSetAttribute(k_groth16_check6, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * 6 * FE_GROUP_WORDS * 4));
  return RIPP_OK;
}
