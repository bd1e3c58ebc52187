// Device-resident GIPA / TIPA / TIPA-with-structured-scalar-message provers and the TIPP Groth16
// aggregation prover.  The four state vectors of a GIPA instance stay in HBM across the log n
// halving rounds; per round only the six commitment values (<= 6 x 576 B) come back to the host
// for the Fiat-Shamir hash, and one 32-byte challenge goes down with the fold launches.
//
// Restates (paths relative to the arkworks-rs/ripp checkout; SURVEY.md §3, App. B):
//   ip_proofs/src/gipa.rs:162-312                      GIPA::prove_with_aux / _prove
//   ip_proofs/src/tipa/mod.rs:176-231,304-337,393-422  TIPA::prove_with_srs_shift + KZG openings
//   ip_proofs/src/tipa/structured_scalar_message.rs:211-268
//   ip_proofs/src/applications/groth16_aggregation.rs:77-160  aggregate_proofs
// Outputs are arkworks `serialize_uncompressed` bytes (what derive(CanonicalSerialize) emits for
// GIPAProof / TIPAProof / TIPAWithSSMProof), so the Rust shim deserialises them directly.
#include "common.cuh"
#include "hash.h"
#include "host_fr.h"

#include <thread>

typedef std::vector<uint8_t> Bytes;

// RIPP_B200_TRACE=1: host wall-clock phase trace on stderr (development aid)
#include <chrono>
static bool trace_on() {
  static const bool v = getenv("RIPP_B200_TRACE") != nullptr;
  return v;
}
static double now_ms() {
  return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ------------------------------------------------------------------------------------------------
// host-side serialisation (ark-serialize 0.4 uncompressed; SURVEY.md App. A-4)
// ------------------------------------------------------------------------------------------------
static void put_fr(Bytes& o, const Fr& m) {
  Fr c = m.from_mont();
  const uint8_t* p = (const uint8_t*)c.v;
  o.insert(o.end(), p, p + 32);
}
static void put_fq_le(Bytes& o, const Fq& m) {
  Fq c = m.from_mont();
  const uint8_t* p = (const uint8_t*)c.v;
  o.insert(o.end(), p, p + 48);
}
static void put_fq_be(Bytes& o, const Fq& m, uint8_t flags = 0) {
  Fq c = m.from_mont();
  const uint8_t* p = (const uint8_t*)c.v;
  size_t at = o.size();
  for (int i = 47; i >= 0; i--) o.push_back(p[i]);
  o[at] |= flags;
}
static void put_gt(Bytes& o, const Fq12& f) {
  const Fq* c = reinterpret_cast<const Fq*>(&f);
  for (int i = 0; i < 12; i++) put_fq_le(o, c[i]);
}
// ark-bls12-381 0.4: big-endian x || y, infinity = 0x40 then zeros
static void put_g1(Bytes& o, const G1Aff& p) {
  if (p.is_inf()) {
    o.push_back(0x40);
    o.insert(o.end(), 95, 0);
    return;
  }
  put_fq_be(o, p.x);
  put_fq_be(o, p.y);
}
static void put_g2(Bytes& o, const G2Aff& p) {
  if (p.is_inf()) {
    o.push_back(0x40);
    o.insert(o.end(), 191, 0);
    return;
  }
  put_fq_be(o, p.x.c1);
  put_fq_be(o, p.x.c0);
  put_fq_be(o, p.y.c1);
  put_fq_be(o, p.y.c0);
}
static void put_u64_le(Bytes& o, uint64_t v) {
  for (int i = 0; i < 8; i++) o.push_back((uint8_t)(v >> (8 * i)));
}
static void put_u64_be(Bytes& o, uint64_t v) {
  for (int i = 7; i >= 0; i--) o.push_back((uint8_t)(v >> (8 * i)));
}

static Fr fr_from_u128_be(const uint8_t* d) {
  // gipa.rs:248-251: Fr::from(u128::from_be_bytes(digest[0..16]))
  Fr c = Fr::zero();
  for (int i = 0; i < 16; i++) c.v[(15 - i) / 4] |= (uint32_t)d[i] << (8 * ((15 - i) % 4));
  return c.to_mont();
}
// ark-ff 0.4 Fp::from_random_bytes: first 32 bytes little-endian, top bit cleared, None if >= r
static bool fr_from_random_bytes(const uint8_t* d, Fr* out) {
  Fr c;
  memcpy(c.v, d, 32);
  c.v[7] &= 0x7fffffffu;
  for (int i = 7; i >= 0; i--) {
    uint32_t m = FrParams::p(i);
    if (c.v[i] < m) break;
    if (c.v[i] > m) return false;
    if (i == 0) return false;  // equal to r
  }
  *out = c.to_mont();
  return true;
}
// tipa/mod.rs:195-209 and friends: hash(nonce_be || parts) until from_random_bytes accepts
static Fr challenge_from_random_bytes(const Bytes& parts) {
  for (uint64_t nonce = 0;; nonce++) {
    Bytes h;
    put_u64_be(h, nonce);
    h.insert(h.end(), parts.begin(), parts.end());
    uint8_t d[64];
    ripp_hash::blake2b512(h.data(), h.size(), d);
    Fr c;
    if (fr_from_random_bytes(d, &c)) return c;
  }
}

// ------------------------------------------------------------------------------------------------
// typed device vectors
// ------------------------------------------------------------------------------------------------
enum VT { VT_NONE = 0, VT_G1 = 1, VT_G2 = 2, VT_FR = 3, VT_GT = 4 };
static size_t vt_size(int t) { return t == VT_G1 ? 96 : t == VT_G2 ? 192 : t == VT_FR ? 32 : t == VT_GT ? 576 : 0; }

struct Slice {
  int t;
  const char* p;
};
static Slice at(int t, const void* base, size_t off) { return Slice{t, base ? (const char*)base + off * vt_size(t) : nullptr}; }

// result of one inner product / commitment, host copy
struct Val {
  int t;  // VT_GT / VT_G1 / VT_G2 / VT_FR
  alignas(16) uint8_t raw[576];
};
static void put_val(Bytes& o, const Val& v) {
  switch (v.t) {
    case VT_GT: put_gt(o, *reinterpret_cast<const Fq12*>(v.raw)); break;
    case VT_G1: put_g1(o, *reinterpret_cast<const G1Aff*>(v.raw)); break;
    case VT_G2: put_g2(o, *reinterpret_cast<const G2Aff*>(v.raw)); break;
    case VT_FR: put_fr(o, *reinterpret_cast<const Fr*>(v.raw)); break;
  }
}

static int ip_out_type(int a, int b) {
  if ((a == VT_G1 && b == VT_G2) || (a == VT_G2 && b == VT_G1)) return VT_GT;
  if (a == VT_NONE || b == VT_NONE) return VT_FR;  // SSMPlaceholderCommitment: Fr::zero()
  if (a == VT_FR && b == VT_FR) return VT_FR;
  return a == VT_FR ? b : a;  // MSM
}

// Up to 8 inner products of equal length evaluated together; pairing-type ones share one launch.
static int eval_products(ripp_ctx* ctx, int k, const Slice* xs, const Slice* ys, size_t n, Val* out) {
  CU(cudaSetDevice(ctx->device));  // the current device is per host thread: worker threads start on device 0
  void* res;
  OK(scratch(ctx, 10, 8 * 576 + 8 * 576, &res));
  char* r = (char*)res;
  const void *g1[8], *g2[8];
  int pair_slot[8], np = 0;
  for (int i = 0; i < k; i++) {
    out[i].t = ip_out_type(xs[i].t, ys[i].t);
    memset(out[i].raw, 0, sizeof(out[i].raw));
    if (out[i].t == VT_GT) {
      bool xg1 = xs[i].t == VT_G1;
      g1[np] = xg1 ? xs[i].p : ys[i].p;
      g2[np] = xg1 ? ys[i].p : xs[i].p;
      pair_slot[np++] = i;
    }
  }
  // children see the state the caller queued on ctx's stream (previous folds) before they start
  for (int j = 0; j < 6; j++)
    if (ctx->child[j]) OK(ripp_fork(ctx, ctx->child[j]));
  // MSM-type products go to child streams FIRST, then the pairing batch on ctx's stream; result copies
  // (which block the host on pageable memory) only after everything has been queued, so the launches overlap
  ripp_ctx* kids[8];
  int kid_of[8];
  int nk = 0;
  for (int i = 0; i < k; i++) {
    int a = xs[i].t, b = ys[i].t;
    kid_of[i] = -1;
    if (out[i].t == VT_GT || a == VT_NONE || b == VT_NONE) continue;
    char* dst = r + 8 * 576 + 576 * i;
    if (a == VT_FR && b == VT_FR) {
      OK(ripp_scalar_ip_dev(ctx, xs[i].p, ys[i].p, n, dst));
      continue;
    }
    ripp_ctx* kid = ripp_child(ctx, nk % 6);
    if (!kid) return fail(RIPP_ERR_CUDA, "child context");
    if (nk >= 6) return fail(RIPP_ERR_ARG, "too many MSM-type products in one batch");
    OK(ripp_fork(ctx, kid));
    kid_of[i] = nk;
    kids[nk++] = kid;
    const char* pts = a == VT_FR ? ys[i].p : xs[i].p;
    const char* sc = a == VT_FR ? xs[i].p : ys[i].p;
    if (out[i].t == VT_G1)
      OK(ripp_msm_g1_dev(kid, pts, sc, n, dst));
    else
      OK(ripp_msm_g2_dev(kid, pts, sc, n, dst));
  }
  if (np) OK(ripp_pairing_batch_l6(ctx, np, g1, g2, n, r, true));
  // results come back through the context's page-locked staging block: MSM-type ones join ctx's stream first, then
  // ONE copy of the whole result block and ONE synchronisation per batch
  uint8_t* pin;
  OK(pinned(ctx, &pin));
  for (int j = 0; j < nk; j++) OK(ripp_join(ctx, kids[j]));
  CU(cudaMemcpyAsync(pin, r, 16 * 576, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < k; i++) {
    int a = xs[i].t, b = ys[i].t;
    if (out[i].t == VT_GT || a == VT_NONE || b == VT_NONE) continue;
    memcpy(out[i].raw, pin + 8 * 576 + 576 * i, vt_size(out[i].t));
  }
  for (int j = 0; j < np; j++) memcpy(out[pair_slot[j]].raw, pin + 576 * j, 576);
  return RIPP_OK;
}

// gipa.rs:235-258 (prover) == :330-353 (verifier): Blake2b-512 over nonce_be(8) || previous c || the six
// commitments of the round; x = u128_be(digest[0..16]); returns (c, c_inv) = (x^-1, x) -- swapped as gipa.rs:253-255.
static void gipa_challenge(const Fr& prev, const Val* com, Fr* c, Fr* c_inv) {
  for (uint64_t nonce = 0;; nonce++) {
    Bytes h;
    put_u64_be(h, nonce);
    put_fr(h, prev);
    for (int i = 0; i < 6; i++) {
      if (i % 3 == 2) put_u64_le(h, 1);  // IdentityOutput<T>(Vec<T>) of length 1
      put_val(h, com[i]);
    }
    uint8_t d[64];
    ripp_hash::blake2b512(h.data(), h.size(), d);
    *c_inv = fr_from_u128_be(d);
    if (!c_inv->is_zero()) {
      *c = c_inv->inv();
      return;
    }
  }
}

// gipa.rs:261-291 for one round: A <- A_R c + A_L, B <- B_R c^-1 + B_L, v <- v_R c^-1 + v_L, w <- w_R c + w_L, in place over
// the lower halves.  Short vectors: ONE fused launch on ctx's stream; long ones: four kernels on four streams.
static int fold_typed(ripp_ctx* ctx, int t, char* base, size_t split, const Fr& c);
// pre: NULL, or the [2^H] images of the upper halves that fold_pre queued (fused launch over precomputed bases)
static int fold_round(ripp_ctx* ctx, const int* types, char* const* bases, size_t split, const Fr& c, const Fr& c_inv,
                      void* const* pre = nullptr) {
  const void *hi[4], *lo[4], *cs[4];
  void* out[4];
  int ty[4];
  const Fr* sc[4] = {&c, &c_inv, &c_inv, &c};
  for (int i = 0; i < 4; i++) {
    ty[i] = (types[i] == VT_NONE || !bases[i]) ? 0 : (types[i] == VT_G1 ? 1 : (types[i] == VT_G2 ? 2 : 3));
    lo[i] = bases[i];
    hi[i] = bases[i] ? bases[i] + split * vt_size(types[i]) : nullptr;
    out[i] = bases[i];
    cs[i] = sc[i]->v;
  }
  int fused = 0;
  OK(ripp_fold4_internal(ctx, ty, hi, lo, cs, split, out, &fused, pre));
  if (fused) return RIPP_OK;
  ripp_ctx* k1 = ripp_child(ctx, 0);
  ripp_ctx* k2 = ripp_child(ctx, 1);
  ripp_ctx* k3 = ripp_child(ctx, 2);
  if (!k1 || !k2 || !k3) return fail(RIPP_ERR_CUDA, "child context");
  OK(ripp_fork(ctx, k1));
  OK(ripp_fork(ctx, k2));
  OK(ripp_fork(ctx, k3));
  OK(fold_typed(ctx, types[0], bases[0], split, c));
  OK(fold_typed(k1, types[1], bases[1], split, c_inv));
  OK(fold_typed(k2, types[2], bases[2], split, c_inv));
  OK(fold_typed(k3, types[3], bases[3], split, c));
  OK(ripp_join(ctx, k1));
  OK(ripp_join(ctx, k2));
  OK(ripp_join(ctx, k3));
  return RIPP_OK;
}

// The challenge-independent half of a short round's folds: D = [2^H] of every G1 / G2 element of the upper halves, queued
// on child 7 (eval_products and fold_round use children 0-5, tipa_prove 5) before the round's products, so that it runs
// in the Miller / final exponentiation / hash window; the caller joins the child before fold_round reads `pre`.
static int fold_pre(ripp_ctx* ctx, const int* types, char* const* bases, size_t split, char* buf, void** pre) {
  int ty[4];
  const void* hi[4];
  size_t off = 0;
  for (int i = 0; i < 4; i++) {
    ty[i] = (types[i] == VT_G1 || types[i] == VT_G2) && bases[i] ? types[i] : 0;
    hi[i] = ty[i] ? bases[i] + split * vt_size(types[i]) : nullptr;
    pre[i] = ty[i] ? buf + off : nullptr;
    if (ty[i]) off += split * vt_size(types[i]);
  }
  ripp_ctx* kid = ripp_child(ctx, 7);
  if (!kid) return fail(RIPP_ERR_CUDA, "child context");
  OK(ripp_fork(ctx, kid));
  return ripp_fold_pre_internal(kid, ty, hi, split, pre);
}

static int fold_typed(ripp_ctx* ctx, int t, char* base, size_t split, const Fr& c) {
  if (t == VT_NONE || !base) return RIPP_OK;  // HomomorphicPlaceholderValue: no-op (identity/mod.rs:18-30)
  char* hi = base + split * vt_size(t);
  if (t == VT_G1) return ripp_g1_fold_dev(ctx, hi, base, c.v, split, base);
  if (t == VT_G2) return ripp_g2_fold_dev(ctx, hi, base, c.v, split, base);
  return ripp_fr_fold_dev(ctx, hi, base, c.v, split, base);
}

// ------------------------------------------------------------------------------------------------
// GIPA (gipa.rs:162-312)
// ------------------------------------------------------------------------------------------------
struct GipaSpec {
  int a, b, v, w;  // element types of the left message, right message, left key, right key
};
static bool gipa_spec(int kind, GipaSpec* s) {
  switch (kind) {
    case RIPP_GIPA_PAIRING: *s = {VT_G1, VT_G2, VT_G2, VT_G1}; return true;
    case RIPP_GIPA_MULTIEXP_PEDERSEN: *s = {VT_G1, VT_FR, VT_G2, VT_G1}; return true;
    case RIPP_GIPA_MULTIEXP_SSM: *s = {VT_G1, VT_FR, VT_G2, VT_NONE}; return true;
    case RIPP_GIPA_SCALAR_PEDERSEN_G2_G2: *s = {VT_FR, VT_FR, VT_G2, VT_G2}; return true;
    case RIPP_GIPA_SCALAR_PEDERSEN_G2_G1: *s = {VT_FR, VT_FR, VT_G2, VT_G1}; return true;
    case RIPP_GIPA_SCALAR_SSM: *s = {VT_FR, VT_FR, VT_G2, VT_NONE}; return true;
    case RIPP_GIPA_SCALAR_SSM_G1: *s = {VT_FR, VT_FR, VT_G1, VT_NONE}; return true;
  }
  return false;
}

struct GipaOut {
  Bytes proof;                 // GIPAProof, serialize_uncompressed
  std::vector<Fr> transcript;  // r_transcript (reversed: element 0 = last round's c)
  Val a0, b0, v0, w0;          // r_base and ck_base
};

// prev0: challenge of the round BEFORE the first one proved here (a sharded prover hands its tail over after its
// own rounds, parallel.py); NULL = a fresh transcript (the default value of gipa.rs:237-238).
// pre_steps / pre_transcript: rounds already proved on LONGER vectors by the sharded prover (sharded.cuh), oldest first;
// the rounds proved here continue that transcript and the emitted proof covers all of them.
static int gipa_prove(ripp_ctx* ctx, const GipaSpec& sp, const void* a_in, const void* b_in, const void* v_in,
                      const void* w_in, size_t n, GipaOut* out, const Fr* prev0 = nullptr,
                      const std::vector<std::vector<Val>>* pre_steps = nullptr, const std::vector<Fr>* pre_transcript = nullptr) {
  if (n == 0 || (n & (n - 1)))
    return fail(RIPP_ERR_NOT_POW2, "left length, right length: " + std::to_string(n) + ", " + std::to_string(n));
  CU(cudaSetDevice(ctx->device));
  // working copies (gipa.rs:175-176 clones all four vectors)
  size_t sa = n * vt_size(sp.a), sb = n * vt_size(sp.b), sv = n * vt_size(sp.v), sw = n * vt_size(sp.w);
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  void* work;
  OK(scratch(ctx, 11, up(sa) + up(sb) + up(sv) + up(sw) + 1024, &work));
  char* A = (char*)work;
  char* B = A + up(sa);
  char* V = B + up(sb);
  char* W = sp.w == VT_NONE ? nullptr : V + up(sv);
  CU(cudaMemcpyAsync(A, a_in, sa, cudaMemcpyDeviceToDevice, ctx->stream));
  CU(cudaMemcpyAsync(B, b_in, sb, cudaMemcpyDeviceToDevice, ctx->stream));
  CU(cudaMemcpyAsync(V, v_in, sv, cudaMemcpyDeviceToDevice, ctx->stream));
  if (W) CU(cudaMemcpyAsync(W, w_in, sw, cudaMemcpyDeviceToDevice, ctx->stream));

  std::vector<std::vector<Val>> steps;  // per round: com_1 (3) then com_2 (3)
  std::vector<Fr> transcript;
  if (pre_steps) steps = *pre_steps;
  if (pre_transcript) transcript = *pre_transcript;
  // [2^H] images of the upper halves for the rounds with split <= pre_max (fold_pre), sized for the first of them
  const size_t pre_max = ripp_fold_pre_max_n();
  char* pre_buf = nullptr;
  if (pre_max && n >= 2) {
    const size_t first = n / 2 < pre_max ? n / 2 : pre_max;
    size_t bytes = 0;
    for (int t : {sp.a, sp.b, sp.v, sp.w})
      if (t == VT_G1 || t == VT_G2) bytes += first * vt_size(t);
    if (bytes) OK(scratch(ctx, 29, bytes, (void**)&pre_buf));
  }
  size_t len = n;
  while (len > 1) {
    size_t split = len / 2;
    const int types[4] = {sp.a, sp.b, sp.v, sp.w};
    char* const bases[4] = {A, B, V, W};
    void* pre[4];
    const bool use_pre = pre_buf && split <= pre_max;
    if (use_pre) OK(fold_pre(ctx, types, bases, split, pre_buf, pre));
    // gipa.rs:209-231 -- com_1 = (IP(A_R, v_L), IP(w_R, B_L), IP(A_R, B_L)); com_2 = (IP(A_L, v_R), IP(w_L, B_R), IP(A_L, B_R))
    Slice xs[6] = {at(sp.a, A, split), at(sp.w, W, split), at(sp.a, A, split), at(sp.a, A, 0), at(sp.w, W, 0), at(sp.a, A, 0)};
    Slice ys[6] = {at(sp.v, V, 0), at(sp.b, B, 0), at(sp.b, B, 0), at(sp.v, V, split), at(sp.b, B, split), at(sp.b, B, split)};
    if (sp.w == VT_NONE) xs[1].t = xs[4].t = VT_NONE;
    std::vector<Val> com(6);
    double t_r0 = now_ms();
    OK(eval_products(ctx, 6, xs, ys, split, com.data()));
    if (split <= 32 && ctx->parent) __atomic_store_n(&ctx->parent->rounds_short, 1, __ATOMIC_RELEASE);
    if (trace_on()) fprintf(stderr, "[trace] gipa(a=%d,b=%d) n'=%zu products+prev folds %.2f ms\n", sp.a, sp.b, split, now_ms() - t_r0);
    // gipa.rs:235-258 -- Fiat-Shamir challenge
    Fr c, c_inv;
    gipa_challenge(transcript.empty() ? (prev0 ? *prev0 : Fr::zero()) : transcript.back(), com.data(), &c, &c_inv);
    // gipa.rs:261-291 -- rescale
    if (use_pre) OK(ripp_join(ctx, ripp_child(ctx, 7)));
    OK(fold_round(ctx, types, bases, split, c, c_inv, use_pre ? pre : nullptr));
    steps.push_back(com);
    transcript.push_back(c);
    len = split;
  }
  // base values
  out->a0.t = sp.a;
  out->b0.t = sp.b;
  out->v0.t = sp.v;
  out->w0.t = sp.w;
  memset(out->a0.raw, 0, 576);
  memset(out->b0.raw, 0, 576);
  memset(out->v0.raw, 0, 576);
  memset(out->w0.raw, 0, 576);
  CU(cudaMemcpyAsync(out->a0.raw, A, vt_size(sp.a), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(out->b0.raw, B, vt_size(sp.b), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(out->v0.raw, V, vt_size(sp.v), cudaMemcpyDeviceToHost, ctx->stream));
  if (W) CU(cudaMemcpyAsync(out->w0.raw, W, vt_size(sp.w), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  // gipa.rs:298-299 -- reversed
  out->transcript.assign(transcript.rbegin(), transcript.rend());
  out->proof.clear();
  put_u64_le(out->proof, steps.size());
  for (size_t r = steps.size(); r-- > 0;) {
    for (int i = 0; i < 6; i++) {
      if (i % 3 == 2) put_u64_le(out->proof, 1);
      put_val(out->proof, steps[r][i]);
    }
  }
  put_val(out->proof, out->a0);
  put_val(out->proof, out->b0);
  return RIPP_OK;
}

static int copy_out(const Bytes& b, uint8_t* dst, size_t cap, size_t* len) {
  if (len) *len = b.size();
  if (!dst || cap < b.size()) return fail(RIPP_ERR_ARG, "output buffer too small: need " + std::to_string(b.size()));
  memcpy(dst, b.data(), b.size());
  return RIPP_OK;
}

extern "C" int ripp_gipa_prove_resume_dev(ripp_ctx* ctx, int kind, const void* a_dev, const void* b_dev, const void* v_dev,
                                          const void* w_dev, size_t n, const void* prev_challenge, uint8_t* proof_out,
                                          size_t proof_cap, size_t* proof_len, void* transcript_out, uint8_t* ck_base_out,
                                          size_t ck_cap, size_t* ck_len) {
  GipaSpec sp;
  if (!ctx || !gipa_spec(kind, &sp)) return fail(RIPP_ERR_ARG, "bad context or GIPA kind");
  if (!a_dev || !b_dev || !v_dev || (sp.w != VT_NONE && !w_dev)) return fail(RIPP_ERR_ARG, "null vector");
  GipaOut g;
  Fr prev;
  if (prev_challenge) memcpy(prev.v, prev_challenge, 32);
  OK(gipa_prove(ctx, sp, a_dev, b_dev, v_dev, w_dev, n, &g, prev_challenge ? &prev : nullptr));
  OK(copy_out(g.proof, proof_out, proof_cap, proof_len));
  if (transcript_out) memcpy(transcript_out, g.transcript.data(), g.transcript.size() * sizeof(Fr));
  Bytes ck;
  put_val(ck, g.v0);
  if (sp.w != VT_NONE) put_val(ck, g.w0);
  return copy_out(ck, ck_base_out, ck_cap, ck_len);
}

// GIPA::prove (gipa.rs:108-133), the checked entry: recompute IP(l, r) and the two message commitments from the
// device vectors, compare them with the caller's statement (`com` = com_a || com_b || com_t in the verifier's
// serialisation; the *_SSM kinds have no right commitment), then prove.  Order of the checks as the reference:
// inner product, power-of-two length, commitments.
extern "C" int ripp_gipa_prove_checked_dev(ripp_ctx* ctx, int kind, const void* a_dev, const void* b_dev, const void* v_dev,
                                           const void* w_dev, size_t n, const uint8_t* com, size_t com_len,
                                           uint8_t* proof_out, size_t proof_cap, size_t* proof_len) {
  GipaSpec sp;
  if (!ctx || !gipa_spec(kind, &sp)) return fail(RIPP_ERR_ARG, "bad context or GIPA kind");
  if (!a_dev || !b_dev || !v_dev || (sp.w != VT_NONE && !w_dev) || !com) return fail(RIPP_ERR_ARG, "null argument");
  // t = IP(a, b); com_a = LMC::commit(v, a) = IP(a, v); com_b = RMC::commit(w, b) = IP(w, b)
  Slice xs[3] = {Slice{sp.a, (const char*)a_dev}, Slice{sp.w, (const char*)w_dev}, Slice{sp.a, (const char*)a_dev}};
  Slice ys[3] = {Slice{sp.v, (const char*)v_dev}, Slice{sp.b, (const char*)b_dev}, Slice{sp.b, (const char*)b_dev}};
  Val got[3];
  if (n) {
    OK(eval_products(ctx, 3, xs, ys, n, got));
  } else {
    for (int i = 0; i < 3; i++) {  // empty products: the neutral element of the output type
      got[i].t = ip_out_type(xs[i].t, ys[i].t);
      memset(got[i].raw, 0, sizeof(got[i].raw));
      if (got[i].t == VT_GT) *reinterpret_cast<Fq12*>(got[i].raw) = Fq12::one();
    }
  }
  Bytes sa, sb, st;
  put_val(sa, got[0]);
  if (sp.w != VT_NONE) put_val(sb, got[1]);
  put_u64_le(st, 1);
  put_val(st, got[2]);
  if (com_len != sa.size() + sb.size() + st.size()) return fail(RIPP_ERR_ARG, "statement has the wrong length for this GIPA kind");
  const uint8_t* c_a = com;
  const uint8_t* c_b = c_a + sa.size();
  const uint8_t* c_t = c_b + sb.size();
  if (memcmp(c_t + 8, st.data() + 8, st.size() - 8) != 0)
    return fail(RIPP_ERR_INNER_PRODUCT, "InnerProductInvalid: IP(l, r) differs from the claimed value (gipa.rs:113-115)");
  if (n == 0 || (n & (n - 1)))
    return fail(RIPP_ERR_NOT_POW2, "left length, right length: " + std::to_string(n) + ", " + std::to_string(n));
  if (memcmp(c_a, sa.data(), sa.size()) != 0 || memcmp(c_b, sb.data(), sb.size()) != 0 || memcmp(c_t, st.data(), 8) != 0)
    return fail(RIPP_ERR_INNER_PRODUCT, "InnerProductInvalid: a commitment does not open to the given message (gipa.rs:123-128)");
  GipaOut g;
  OK(gipa_prove(ctx, sp, a_dev, b_dev, v_dev, w_dev, n, &g));
  return copy_out(g.proof, proof_out, proof_cap, proof_len);
}

extern "C" int ripp_gipa_prove_dev(ripp_ctx* ctx, int kind, const void* a_dev, const void* b_dev, const void* v_dev,
                                   const void* w_dev, size_t n, uint8_t* proof_out, size_t proof_cap, size_t* proof_len,
                                   void* transcript_out, uint8_t* ck_base_out, size_t ck_cap, size_t* ck_len) {
  GipaSpec sp;
  if (!ctx || !gipa_spec(kind, &sp)) return fail(RIPP_ERR_ARG, "bad context or GIPA kind");
  if (!a_dev || !b_dev || !v_dev || (sp.w != VT_NONE && !w_dev)) return fail(RIPP_ERR_ARG, "null vector");
  GipaOut g;
  OK(gipa_prove(ctx, sp, a_dev, b_dev, v_dev, w_dev, n, &g));
  OK(copy_out(g.proof, proof_out, proof_cap, proof_len));
  if (transcript_out) memcpy(transcript_out, g.transcript.data(), g.transcript.size() * sizeof(Fr));
  Bytes ck;
  put_val(ck, g.v0);
  if (sp.w != VT_NONE) put_val(ck, g.w0);
  return copy_out(ck, ck_base_out, ck_cap, ck_len);
}

// ------------------------------------------------------------------------------------------------
// KZG opening of a structured final commitment key (tipa/mod.rs:304-337, 407-422)
// ------------------------------------------------------------------------------------------------
// coefficients of f(X) = prod_j (1 + x_j r^(2^j) X^(2^(j+1))) interleaved with zeros (length 2n-1),
// then q = (f - f(z)) / (X - z) by synthetic division; returns q zero-padded to n_srs (Montgomery).
static std::vector<Fr> kzg_quotient(const std::vector<Fr>& transcript, const Fr& r_shift, const Fr& z, size_t n_srs) {
  namespace H = hostfr;  // 64-bit-limb host arithmetic: 3 n products per opening (n = 4096: 3.3 ms -> 0.3 ms)
  std::vector<Fr> coeffs(1, Fr::one());
  Fr power_2_r = r_shift;
  for (size_t i = 0; i < transcript.size(); i++) {
    Fr m = H::mul(transcript[i], power_2_r);
    size_t cur = coeffs.size();
    coeffs.reserve(2 * cur);
    for (size_t j = 0; j < cur; j++) coeffs.push_back(H::mul(coeffs[j], m));
    power_2_r = H::mul(power_2_r, power_2_r);
  }
  // f has degree 2(len-1): f[2i] = coeffs[i], odd coefficients are zero
  size_t deg = 2 * (coeffs.size() - 1);
  std::vector<Fr> q(n_srs, Fr::zero());
  Fr carry = Fr::zero();
  for (size_t i = deg; i >= 1; i--) {
    carry = H::mul(z, carry);
    if (i % 2 == 0) carry = H::add(coeffs[i / 2], carry);
    q[i - 1] = carry;
  }
  return q;
}

// The quotient coefficients alone (host in, host out): the sharded KZG opening lets every rank run the MSM over
// its slice of the SRS powers (SURVEY.md §8e "KZG openings").
extern "C" int ripp_kzg_quotient(const void* transcript, size_t k, const void* r_shift, const void* z, size_t n_srs,
                                 void* fr_out) {
  if (!transcript || !r_shift || !z || !fr_out) return fail(RIPP_ERR_ARG, "null argument");
  if (n_srs != 2 * ((size_t)1 << k) - 1) return fail(RIPP_ERR_ARG, "SRS length must be 2*2^k - 1");
  std::vector<Fr> t(k);
  memcpy(t.data(), transcript, k * sizeof(Fr));
  Fr rs, zz;
  memcpy(rs.v, r_shift, 32);
  memcpy(zz.v, z, 32);
  std::vector<Fr> q = kzg_quotient(t, rs, zz, n_srs);
  memcpy(fr_out, q.data(), n_srs * sizeof(Fr));
  return RIPP_OK;
}

template <class F>
static int kzg_open(ripp_ctx* ctx, const void* srs_dev, size_t n_srs, const std::vector<Fr>& transcript, const Fr& r_shift,
                    const Fr& z, Aff<F>* out_host) {
  CU(cudaSetDevice(ctx->device));  // may run on a worker thread (tipa_prove)
  double t_q0 = now_ms();
  std::vector<Fr> q = kzg_quotient(transcript, r_shift, z, n_srs);
  if (trace_on()) fprintf(stderr, "[trace] kzg quotient (host, %zu coefficients) %.2f ms\n", n_srs, now_ms() - t_q0);
  void* d;
  OK(scratch(ctx, 12, n_srs * sizeof(Fr) + 1024, &d));
  CU(cudaMemcpyAsync(d, q.data(), n_srs * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
  char* res = (char*)d + ((n_srs * sizeof(Fr) + 255) & ~(size_t)255);
  if (sizeof(F) == sizeof(Fq))
    OK(ripp_msm_g1_dev(ctx, srs_dev, d, n_srs, res));
  else
    OK(ripp_msm_g2_dev(ctx, srs_dev, d, n_srs, res));
  CU(cudaMemcpyAsync(out_host, res, sizeof(Aff<F>), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

extern "C" int ripp_kzg_open_g1_dev(ripp_ctx* ctx, const void* srs_g1_dev, size_t n_srs, const void* transcript, size_t k,
                                    const void* r_shift, const void* z, void* g1_aff_out) {
  if (!ctx || !srs_g1_dev || !transcript || !r_shift || !z || !g1_aff_out) return fail(RIPP_ERR_ARG, "null argument");
  if (n_srs != 2 * ((size_t)1 << k) - 1) return fail(RIPP_ERR_ARG, "SRS length must be 2*2^k - 1");
  std::vector<Fr> t(k);
  memcpy(t.data(), transcript, k * sizeof(Fr));
  Fr rs, zz;
  memcpy(rs.v, r_shift, 32);
  memcpy(zz.v, z, 32);
  return kzg_open<Fq>(ctx, srs_g1_dev, n_srs, t, rs, zz, (G1Aff*)g1_aff_out);
}
extern "C" int ripp_kzg_open_g2_dev(ripp_ctx* ctx, const void* srs_g2_dev, size_t n_srs, const void* transcript, size_t k,
                                    const void* r_shift, const void* z, void* g2_aff_out) {
  if (!ctx || !srs_g2_dev || !transcript || !r_shift || !z || !g2_aff_out) return fail(RIPP_ERR_ARG, "null argument");
  if (n_srs != 2 * ((size_t)1 << k) - 1) return fail(RIPP_ERR_ARG, "SRS length must be 2*2^k - 1");
  std::vector<Fr> t(k);
  memcpy(t.data(), transcript, k * sizeof(Fr));
  Fr rs, zz;
  memcpy(rs.v, r_shift, 32);
  memcpy(zz.v, z, 32);
  return kzg_open<Fq2>(ctx, srs_g2_dev, n_srs, t, rs, zz, (G2Aff*)g2_aff_out);
}

// ------------------------------------------------------------------------------------------------
// TIPA (tipa/mod.rs:176-231) and TIPA with structured scalar message (structured_scalar_message.rs:211-268)
// ------------------------------------------------------------------------------------------------
// srs_g1 = g^{alpha^i}, srs_g2 = h^{beta^i}, i < 2n-1, device resident (tipa/mod.rs:96-111).
static int tipa_prove(ripp_ctx* ctx, int kind, const void* srs_g1, const void* srs_g2, const void* a, const void* b,
                      const void* v, const void* w, size_t n, const Fr& r_shift, Bytes* proof) {
  GipaSpec sp;
  if (!gipa_spec(kind, &sp)) return fail(RIPP_ERR_ARG, "bad GIPA kind");
  if (sp.v != VT_G2 || (sp.w != VT_G1 && sp.w != VT_NONE)) return fail(RIPP_ERR_ARG, "TIPA needs keys in (G2, G1)");
  // the reference panics on `transcript.first().unwrap()` for a length-1 instance (tipa/mod.rs:199)
  if (n < 2) return fail(RIPP_ERR_ARG, "TIPA needs at least two elements (the KZG challenge hashes the last round's challenge)");
  if (!srs_g2 || (sp.w != VT_NONE && (!srs_g1 || !w))) return fail(RIPP_ERR_ARG, "null SRS or right key");
  GipaOut g;
  double t_g0 = now_ms();
  OK(gipa_prove(ctx, sp, a, b, v, w, n, &g));
  double t_g1 = now_ms();
  size_t n_srs = 2 * n - 1;
  std::vector<Fr> tinv(g.transcript.size());
  for (size_t i = 0; i < tinv.size(); i++) tinv[i] = g.transcript[i].inv();
  // KZG challenge (tipa/mod.rs:195-209 / structured_scalar_message.rs:238-251)
  Bytes parts;
  put_fr(parts, g.transcript[0]);
  put_val(parts, g.v0);
  if (sp.w != VT_NONE) put_val(parts, g.w0);
  Fr c = challenge_from_random_bytes(parts);
  G2Aff open_a;
  G1Aff open_b;
  Fr shift_a = sp.w != VT_NONE ? r_shift.inv() : Fr::one();  // SSM variant opens with shift 1
  int st_b = RIPP_OK;
  std::string err_b;
  std::thread tb;
  if (sp.w != VT_NONE) {  // the G1 opening runs on a child context from a second host thread
    ripp_ctx* kid = ripp_child(ctx, 5);
    if (!kid) return fail(RIPP_ERR_CUDA, "child context");
    OK(ripp_fork(ctx, kid));
    tb = std::thread([&, kid] {
      st_b = kzg_open<Fq>(kid, srs_g1, n_srs, g.transcript, Fr::one(), c, &open_b);
      if (st_b != RIPP_OK) err_b = ripp_err_slot();
    });
  }
  int st_a = kzg_open<Fq2>(ctx, srs_g2, n_srs, tinv, shift_a, c, &open_a);
  if (tb.joinable()) tb.join();
  if (st_a != RIPP_OK) return st_a;
  if (st_b != RIPP_OK) return fail(st_b, err_b);
  *proof = g.proof;
  put_val(*proof, g.v0);
  if (sp.w != VT_NONE) {
    put_val(*proof, g.w0);
    put_g2(*proof, open_a);
    put_g1(*proof, open_b);
  } else {
    put_g2(*proof, open_a);
  }
  if (trace_on()) fprintf(stderr, "[trace] tipa kind=%d: gipa %.2f ms, kzg openings %.2f ms\n", kind, t_g1 - t_g0, now_ms() - t_g1);
  return RIPP_OK;
}

extern "C" int ripp_tipa_prove_dev(ripp_ctx* ctx, int kind, const void* srs_g1_dev, const void* srs_g2_dev, const void* a_dev,
                                   const void* b_dev, const void* v_dev, const void* w_dev, size_t n, const void* r_shift,
                                   uint8_t* proof_out, size_t proof_cap, size_t* proof_len) {
  if (!ctx || !srs_g2_dev || !a_dev || !b_dev || !v_dev) return fail(RIPP_ERR_ARG, "null argument");
  Fr rs = Fr::one();
  if (r_shift) memcpy(rs.v, r_shift, 32);
  Bytes proof;
  OK(tipa_prove(ctx, kind, srs_g1_dev, srs_g2_dev, a_dev, b_dev, v_dev, w_dev, n, rs, &proof));
  return copy_out(proof, proof_out, proof_cap, proof_len);
}

// ------------------------------------------------------------------------------------------------
// TIPP Groth16 aggregation (applications/groth16_aggregation.rs:77-160)
// ------------------------------------------------------------------------------------------------
__global__ void k_fr_powers(Fr r, size_t n, Fr* __restrict__ pw, Fr* __restrict__ pw_inv, Fr r_inv, size_t stride = 1,
                            size_t offset = 0) {
  // r^e and r^-e, e = i stride + offset, by square-and-multiply on the exponent (n threads, log products each)
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fr acc = Fr::one(), acci = Fr::one(), b = r, bi = r_inv;
  for (size_t e = i * stride + offset; e; e >>= 1) {
    if (e & 1) {
      acc = acc * b;
      acci = acci * bi;
    }
    b = b * b;
    bi = bi * bi;
  }
  pw[i] = acc;
  pw_inv[i] = acci;
}
template <class T>
__global__ void k_gather_stride2(const T* __restrict__ in, size_t n, T* __restrict__ out, size_t stride = 2, size_t offset = 0) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = in[i * stride + offset];
}

extern "C" int ripp_tipp_aggregate_dev(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, const void* a_dev,
                                       const void* b_dev, const void* c_dev, size_t n, uint8_t* proof_out, size_t proof_cap,
                                       size_t* proof_len) {
  if (!ctx || !srs_g1_dev || !srs_g2_dev || !a_dev || !b_dev || !c_dev) return fail(RIPP_ERR_ARG, "null argument");
  if (n == 0 || (n & (n - 1))) return fail(RIPP_ERR_NOT_POW2, "number of proofs must be a power of two");
  if (n < 2) return fail(RIPP_ERR_ARG, "aggregation needs at least two proofs (tipa/mod.rs:199 unwraps the first challenge)");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  // layout of the aggregation workspace
  void* ws;
  size_t o_ck1 = 0, o_ck2 = o_ck1 + n * 192, o_ar = o_ck2 + n * 96, o_ck1r = o_ar + n * 96, o_pw = o_ck1r + n * 192,
         o_pwi = o_pw + n * 32, o_res = o_pwi + n * 32;
  OK(scratch(ctx, 13, o_res + 8 * 576, &ws));
  char* W = (char*)ws;
  unsigned nb = (unsigned)((n + 127) / 128);
  double t_a0 = now_ms();
  // :98 commitment keys = even SRS powers (tipa/mod.rs:114-118)
  k_gather_stride2<G2Aff><<<nb, 128, 0, st>>>((const G2Aff*)srs_g2_dev, n, (G2Aff*)(W + o_ck1));
  LAUNCHED(ctx);
  k_gather_stride2<G1Aff><<<nb, 128, 0, st>>>((const G1Aff*)srs_g1_dev, n, (G1Aff*)(W + o_ck2));
  LAUNCHED(ctx);
  const void* ck1 = W + o_ck1;
  const void* ck2 = W + o_ck2;
  // :100-102 com_a = IP(a, ck_1), com_b = IP(ck_2, b), com_c = IP(c, ck_1)
  Val com[3];
  {
    Slice xs[3] = {Slice{VT_G1, (const char*)a_dev}, Slice{VT_G1, (const char*)ck2}, Slice{VT_G1, (const char*)c_dev}};
    Slice ys[3] = {Slice{VT_G2, (const char*)ck1}, Slice{VT_G2, (const char*)b_dev}, Slice{VT_G2, (const char*)ck1}};
    OK(eval_products(ctx, 3, xs, ys, n, com));
  }
  // :105-116 r
  Bytes parts;
  for (int i = 0; i < 3; i++) put_val(parts, com[i]);
  Fr r = challenge_from_random_bytes(parts);
  Fr r_inv = r.inv();
  // :118-131 r_vec, a_r = a * r^i, ck_1_r = ck_1 * r^-i
  k_fr_powers<<<nb, 128, 0, st>>>(r, n, (Fr*)(W + o_pw), (Fr*)(W + o_pwi), r_inv);
  LAUNCHED(ctx);
  ripp_ctx* pk = ripp_child(ctx, 5);
  if (!pk) return fail(RIPP_ERR_CUDA, "child context");
  OK(ripp_fork(ctx, pk));
  OK(ripp_g2_scale_dev(pk, ck1, W + o_pwi, n, W + o_ck1r));   // the long one (G2, 255-bit) on its own stream
  OK(ripp_g1_scale_dev(ctx, a_dev, W + o_pw, n, W + o_ar));
  // :125 agg_c = MSM(c, r_vec) needs only r_vec: queue it behind the G1 scaling on a third stream
  ripp_ctx* mk = ripp_child(ctx, 4);
  if (!mk) return fail(RIPP_ERR_CUDA, "child context");
  OK(ripp_fork(ctx, mk));
  OK(ripp_msm_g1_dev(mk, c_dev, W + o_pw, n, W + o_res));
  OK(ripp_join(ctx, pk));
  // :124 ip_ab = IP(a_r, b) and the :133-136 sanity product IP(a_r, ck_1_r) are not inputs of the two TIPA
  // proofs: they run from a third host thread on their own child context, overlapping the first GIPA rounds.
  Val ipv[2];
  Val agg_c;
  agg_c.t = VT_G1;
  memset(agg_c.raw, 0, 576);
  int st_ip = RIPP_OK, st_c = RIPP_OK, st_a = RIPP_OK;
  std::string err_ip, err_c;
  // :138-149 the two TIPA proofs are independent as well: three host threads on three child contexts, so the
  // (latency-bound) rounds of both recursions and the two big products overlap on the GPU.  All children are
  // created and forked before any thread starts; after that, failures are reported through the status words.
  ripp_ctx* ik = ripp_child(ctx, 3);
  ripp_ctx* ka = ripp_child(ctx, 6);
  ripp_ctx* kc = ripp_child(ctx, 7);
  if (!ik || !ka || !kc) return fail(RIPP_ERR_CUDA, "child context");
  OK(ripp_fork(ctx, ik));
  OK(ripp_fork(ctx, ka));
  OK(ripp_fork(ctx, kc));
  if (trace_on()) fprintf(stderr, "[trace] aggregate prologue (3 commitments, r, scalings queued) %.2f ms\n", now_ms() - t_a0);
  Bytes proof_ab, proof_c;
  {
    __atomic_store_n(&ctx->rounds_short, 0, __ATOMIC_RELEASE);
    ik->background = 1;
    kc->background = getenv("RIPP_B200_SSM_FOREGROUND") ? 0 : 1;  // the SSM recursion has slack: its long rounds yield CTAs to the pairing recursion
    std::thread tip([&] {
      // 2 n pairs that nothing waits for: started once the pairing recursion has left its long (throughput-bound) rounds
      while (!__atomic_load_n(&ctx->rounds_short, __ATOMIC_ACQUIRE)) std::this_thread::sleep_for(std::chrono::microseconds(20));
      Slice xs[2] = {Slice{VT_G1, W + o_ar}, Slice{VT_G1, W + o_ar}};
      Slice ys[2] = {Slice{VT_G2, (const char*)b_dev}, Slice{VT_G2, W + o_ck1r}};
      st_ip = eval_products(ik, 2, xs, ys, n, ipv);
      if (st_ip != RIPP_OK) err_ip = ripp_err_slot();
    });
    std::thread tc([&] {
      st_c = tipa_prove(kc, RIPP_GIPA_MULTIEXP_SSM, srs_g1_dev, srs_g2_dev, c_dev, W + o_pw, ck1, nullptr, n, Fr::one(), &proof_c);
      if (st_c != RIPP_OK) err_c = ripp_err_slot();
    });
    st_a = tipa_prove(ka, RIPP_GIPA_PAIRING, srs_g1_dev, srs_g2_dev, W + o_ar, b_dev, W + o_ck1r, ck2, n, r, &proof_ab);
    __atomic_store_n(&ctx->rounds_short, 1, __ATOMIC_RELEASE);  // n < 2 or a failed recursion never reaches the short rounds
    tc.join();
    tip.join();
    ik->background = kc->background = 0;  // the children are cached on the context: other entry points get them unhinted
  }
  if (st_a != RIPP_OK) return st_a;
  if (st_c != RIPP_OK) return fail(st_c, err_c);
  if (st_ip != RIPP_OK) return fail(st_ip, err_ip);
  OK(ripp_join(ctx, ka));
  OK(ripp_join(ctx, kc));
  OK(ripp_join(ctx, ik));
  if (memcmp(ipv[1].raw, com[0].raw, 576) != 0)
    return fail(RIPP_ERR_INNER_PRODUCT, "com_a != IP(a_r, ck_1_r) (groth16_aggregation.rs:133-136)");
  // :125 agg_c = MSM(c, r_vec), queued in the prologue on its own stream
  OK(ripp_join(ctx, mk));
  CU(cudaMemcpyAsync(agg_c.raw, W + o_res, 96, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  // AggregateProof { com_a, com_b, com_c, ip_ab, agg_c, tipa_proof_ab, tipa_proof_c } (:58-66)
  Bytes out;
  for (int i = 0; i < 3; i++) put_val(out, com[i]);
  put_val(out, ipv[0]);
  put_val(out, agg_c);
  out.insert(out.end(), proof_ab.begin(), proof_ab.end());
  out.insert(out.end(), proof_c.begin(), proof_c.end());
  return copy_out(out, proof_out, proof_cap, proof_len);
}

extern "C" int ripp_tipp_aggregate(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, const void* a_host,
                                   const void* b_host, const void* c_host, size_t n, uint8_t* proof_out, size_t proof_cap,
                                   size_t* proof_len) {
  if (!ctx || !a_host || !b_host || !c_host) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  void* d;
  OK(scratch(ctx, 14, n * (96 + 192 + 96) + 1024, &d));
  char* p = (char*)d;
  CU(cudaMemcpyAsync(p, a_host, n * 96, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(p + n * 96, c_host, n * 96, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(p + n * 192, b_host, n * 192, cudaMemcpyHostToDevice, ctx->stream));
  return ripp_tipp_aggregate_dev(ctx, srs_g1_dev, srs_g2_dev, p, p + n * 192, p + n * 96, n, proof_out, proof_cap, proof_len);
}

// ------------------------------------------------------------------------------------------------
// SIPP (sipp/src/lib.rs:42-106, 184-224; FiatShamirRng sipp/src/rng.rs:12-73), D = Blake2s
// ------------------------------------------------------------------------------------------------
struct SippRng {
  uint8_t seed[32];
  void init(const Bytes& material) { ripp_hash::blake2s256(material.data(), material.size(), seed); }
  // seed = D(new || seed); the ChaCha20 stream restarts from block 0 with the new key (rng.rs:64-72)
  void absorb(const Bytes& fresh) {
    Bytes b(fresh);
    b.insert(b.end(), seed, seed + 32);
    ripp_hash::blake2s256(b.data(), b.size(), seed);
  }
  // u128::rand = next_u64() | next_u64() << 64 = first 16 keystream bytes, little-endian (lib.rs:85)
  Fr next_u128() const {
    uint8_t ks[64];
    ripp_hash::chacha20_block(seed, 0, ks);
    Fr c = Fr::zero();
    memcpy(c.v, ks, 16);
    return c.to_mont();
  }
};

// product_of_pairings_with_coeffs (sipp/src/lib.rs:184-217): prod e(r_i a_i, b_i); affine host inputs
extern "C" int ripp_sipp_product_with_coeffs(ripp_ctx* ctx, const void* a_aff, const void* b_aff, const void* r, size_t n,
                                             void* gt_out) {
  if (!ctx || !gt_out || (n && (!a_aff || !b_aff || !r))) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  void* d;
  OK(scratch(ctx, 14, n * (96 + 192 + 32 + 96) + 2048, &d));
  char* A = (char*)d;
  char* Bp = A + n * 96;
  char* Rp = Bp + n * 192;
  char* AR = Rp + n * 32;
  char* out = AR + n * 96;
  CU(cudaMemcpyAsync(A, a_aff, n * 96, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(Bp, b_aff, n * 192, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(Rp, r, n * 32, cudaMemcpyHostToDevice, ctx->stream));
  OK(ripp_g1_scale_dev(ctx, A, Rp, n, AR));
  OK(ripp_pairing_ip_dev(ctx, AR, Bp, n, out));
  CU(cudaMemcpyAsync(gt_out, out, 576, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

// SIPP::prove.  a: n G1 affine, b: n G2 affine, r: n Fr, value: GT (all host, Montgomery limbs).
// proof_out: log2(n) pairs (z_l, z_r), each GT serialize_uncompressed (2 * 576 B per round).
extern "C" int ripp_sipp_prove(ripp_ctx* ctx, const void* a_aff, const void* b_aff, const void* r, size_t n,
                               const void* value_gt, uint8_t* proof_out, size_t proof_cap, size_t* proof_len) {
  if (!ctx || !a_aff || !b_aff || !r || !value_gt) return fail(RIPP_ERR_ARG, "null argument");
  if (n == 0 || (n & (n - 1))) return fail(RIPP_ERR_NOT_POW2, "SIPP needs a power-of-two length");
  CU(cudaSetDevice(ctx->device));
  // lib.rs:56-60: rng seeded with the uncompressed serialisation of (a, b, r, value)
  SippRng rng;
  {
    Bytes seed;
    const G1Aff* a = (const G1Aff*)a_aff;
    const G2Aff* b = (const G2Aff*)b_aff;
    const Fr* rr = (const Fr*)r;
    put_u64_le(seed, n);
    for (size_t i = 0; i < n; i++) put_g1(seed, a[i]);
    put_u64_le(seed, n);
    for (size_t i = 0; i < n; i++) put_g2(seed, b[i]);
    put_u64_le(seed, n);
    for (size_t i = 0; i < n; i++) put_fr(seed, rr[i]);
    put_gt(seed, *(const Fq12*)value_gt);
    rng.init(seed);
  }
  void* d;
  OK(scratch(ctx, 14, n * (96 + 192 + 32 + 96) + 4096, &d));
  char* A0 = (char*)d;
  char* Bv = A0 + n * 96;
  char* Rp = Bv + n * 192;
  char* Av = Rp + n * 32;
  char* res = Av + n * 96;
  CU(cudaMemcpyAsync(A0, a_aff, n * 96, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(Bv, b_aff, n * 192, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(Rp, r, n * 32, cudaMemcpyHostToDevice, ctx->stream));
  OK(ripp_g1_scale_dev(ctx, A0, Rp, n, Av));  // lib.rs:61-66: a_i <- a_i r_i
  Bytes proof;
  size_t len = n;
  while (len != 1) {
    len /= 2;
    // lib.rs:77-78: z_l = prod e(a_R, b_L), z_r = prod e(a_L, b_R)
    const void* g1[2] = {Av + len * 96, Av};
    const void* g2[2] = {Bv, Bv + len * 192};
    OK(ripp_pairing_batch_l6(ctx, 2, g1, g2, len, res, true));
    Fq12 z[2];
    CU(cudaMemcpyAsync(z, res, 2 * 576, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    Bytes buf;
    put_gt(buf, z[0]);
    put_gt(buf, z[1]);
    proof.insert(proof.end(), buf.begin(), buf.end());
    rng.absorb(buf);                 // lib.rs:80-84
    Fr x = rng.next_u128();          // lib.rs:85
    Fr x_inv = x.inv();
    // lib.rs:87-100: a <- a_R x + a_L ; b <- b_R x^-1 + b_L   (on two streams)
    {
      const int ty[4] = {1, 2, 0, 0};
      const void* hi[4] = {Av + len * 96, Bv + len * 192, nullptr, nullptr};
      const void* lo[4] = {Av, Bv, nullptr, nullptr};
      const void* cs[4] = {x.v, x_inv.v, nullptr, nullptr};
      void* outp[4] = {Av, Bv, nullptr, nullptr};
      int fused = 0;
      OK(ripp_fold4_internal(ctx, ty, hi, lo, cs, len, outp, &fused));  // both folds in one launch when short enough
      if (!fused) {
        ripp_ctx* kid = ripp_child(ctx, 0);
        if (!kid) return fail(RIPP_ERR_CUDA, "child context");
        OK(ripp_fork(ctx, kid));
        OK(ripp_g1_fold_dev(ctx, Av + len * 96, Av, x.v, len, Av));
        OK(ripp_g2_fold_dev(kid, Bv + len * 192, Bv, x_inv.v, len, Bv));
        OK(ripp_join(ctx, kid));
      }
    }
  }
  CU(cudaStreamSynchronize(ctx->stream));
  return copy_out(proof, proof_out, proof_cap, proof_len);
}

#include "verify.cuh"
#include "verify_batch.cuh"
#include "poly_commit.cuh"
#include "aggregate_batch.cuh"
#include "pc_batch.cuh"
#include "pc_verify_batch.cuh"
#include "sharded.cuh"
