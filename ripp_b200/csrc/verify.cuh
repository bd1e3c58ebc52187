// Verifiers of the inner-product arguments on the GPU (SURVEY.md §8 rows a13, a17, a20, a22; §8f-1).
// Part of the gipa.cu translation unit (shares its serialisation helpers, typed values and eval_products).
//
// Restates (paths relative to the arkworks-rs/ripp checkout):
//   ip_proofs/src/gipa.rs:135-160, 322-415                    GIPA::verify and its three helpers
//   ip_proofs/src/tipa/mod.rs:242-301, 340-370, 393-405        TIPA::verify_with_srs_shift + KZG checks
//   ip_proofs/src/tipa/structured_scalar_message.rs:86-127     GIPAWithSSM::verify_with_structured_scalar_message
//   ip_proofs/src/tipa/structured_scalar_message.rs:270-331    TIPAWithSSM::verify_with_structured_scalar_message
//   ip_proofs/src/applications/groth16_aggregation.rs:162-231  verify_aggregate_proof
//   sipp/src/lib.rs:109-180                                    SIPP::verify
//
// Shape of the work: the Fiat-Shamir chain of a verifier depends only on bytes of the proof, so all
// challenges are recomputed on the host first; the recursive commitment update
//   com <- c com_1 + com + c^-1 com_2   (gipa.rs:355-357, log n times)
// then collapses into ONE multi-exponentiation per commitment component over 2 log n + 1 elements
// (GT: k_gt_pow6 + product tree; G1/G2: the MSM kernels; Fr: host), the final commitment keys are one MSM
// over the key vector (the reference's naive sum, gipa.rs:383 "TODO use MSM"), and every remaining check is
// an inner product of length-1 vectors evaluated by the same kernels the prover uses.
// Inputs are arkworks serialize_uncompressed bytes, as the provers emit them.  Decoding validates exactly what
// ark-serialize's `deserialize_uncompressed` (Valid::check) validates: canonical field encodings, curve membership
// (host, while parsing) and membership of the prime-order subgroups of G1 / G2 / GT (one batch of GPU checks over
// every decoded element, `validate_subgroups`, before any of them reaches the endomorphism-based MSM / fold
// kernels, whose GLV / GLS maps are scalar multiplications only inside the r-torsion).
#pragma once
#include "serde.cuh"

// ------------------------------------------------------------------------------------------------
// decoding (inverse of the put_* helpers; ark-serialize 0.4 uncompressed, SURVEY.md App. A-4)
// ------------------------------------------------------------------------------------------------
struct Reader {
  const uint8_t* p;
  size_t n, off;
  bool ok;
  // every group element decoded from these bytes, for the subgroup checks
  std::vector<G1Aff> g1s;
  std::vector<G2Aff> g2s;
  std::vector<Fq12> gts;
  Reader(const void* data, size_t len) : p((const uint8_t*)data), n(len), off(0), ok(data != nullptr || len == 0) {}
  const uint8_t* take(size_t k) {
    if (!ok || n - off < k) {
      ok = false;
      return nullptr;
    }
    const uint8_t* r = p + off;
    off += k;
    return r;
  }
  bool done() const { return ok && off == n; }
};

template <class P>
static bool canonical_lt_modulus(const uint32_t* v) {
  for (int i = P::N - 1; i >= 0; i--) {
    if (v[i] < P::p(i)) return true;
    if (v[i] > P::p(i)) return false;
  }
  return false;
}
static bool get_fr(Reader& r, Fr* out) {
  const uint8_t* s = r.take(32);
  if (!s) return false;
  Fr c;
  memcpy(c.v, s, 32);
  if (!canonical_lt_modulus<FrParams>(c.v)) return r.ok = false;
  *out = c.to_mont();
  return true;
}
static bool get_fq_le(Reader& r, Fq* out) {
  const uint8_t* s = r.take(48);
  if (!s) return false;
  Fq c;
  memcpy(c.v, s, 48);
  if (!canonical_lt_modulus<FqParams>(c.v)) return r.ok = false;
  *out = c.to_mont();
  return true;
}
// big-endian, the three top bits of the first byte are flags (compressed, infinity, sign)
static bool get_fq_be(Reader& r, Fq* out, uint8_t* flags) {
  const uint8_t* s = r.take(48);
  if (!s) return false;
  uint8_t b[48];
  for (int i = 0; i < 48; i++) b[i] = s[47 - i];
  if (flags) {
    *flags = b[47] & 0xe0;
    b[47] &= 0x1f;
  }
  Fq c;
  memcpy(c.v, b, 48);
  if (!canonical_lt_modulus<FqParams>(c.v)) return r.ok = false;
  *out = c.to_mont();
  return true;
}
static bool get_u64_le(Reader& r, uint64_t* v) {
  const uint8_t* s = r.take(8);
  if (!s) return false;
  *v = 0;
  for (int i = 0; i < 8; i++) *v |= (uint64_t)s[i] << (8 * i);
  return true;
}
static bool get_gt(Reader& r, Fq12* f) {
  Fq* c = reinterpret_cast<Fq*>(f);
  for (int i = 0; i < 12; i++)
    if (!get_fq_le(r, &c[i])) return false;
  r.gts.push_back(*f);
  return true;
}
static Fq fq_small(int k) {
  Fq r = Fq::zero();
  for (int i = 0; i < k; i++) r = r + Fq::one();
  return r;
}
static bool get_g1(Reader& r, G1Aff* p) {
  uint8_t fl = 0;
  Fq x, y;
  if (!get_fq_be(r, &x, &fl) || !get_fq_be(r, &y, nullptr)) return false;
  if (fl & 0x80) return r.ok = false;  // compressed encoding
  if (fl & 0x40) {
    if (!x.is_zero() || !y.is_zero()) return r.ok = false;
    *p = G1Aff::inf();
    return true;
  }
  if (y.sqr() != x.sqr() * x + fq_small(4)) return r.ok = false;  // y^2 = x^3 + 4
  *p = G1Aff{x, y};
  r.g1s.push_back(*p);
  return true;
}
static bool get_g2(Reader& r, G2Aff* p) {
  uint8_t fl = 0;
  Fq2 x, y;
  if (!get_fq_be(r, &x.c1, &fl) || !get_fq_be(r, &x.c0, nullptr) || !get_fq_be(r, &y.c1, nullptr) ||
      !get_fq_be(r, &y.c0, nullptr))
    return false;
  if (fl & 0x80) return r.ok = false;
  if (fl & 0x40) {
    if (!x.is_zero() || !y.is_zero()) return r.ok = false;
    *p = G2Aff::inf();
    return true;
  }
  Fq four = fq_small(4);
  if (y.sqr() != x.sqr() * x + Fq2{four, four}) return r.ok = false;  // y^2 = x^3 + 4 (1 + u)
  *p = G2Aff{x, y};
  r.g2s.push_back(*p);
  return true;
}
static bool get_val(Reader& r, int t, Val* v) {
  v->t = t;
  memset(v->raw, 0, sizeof(v->raw));
  switch (t) {
    case VT_GT: return get_gt(r, reinterpret_cast<Fq12*>(v->raw));
    case VT_G1: return get_g1(r, reinterpret_cast<G1Aff*>(v->raw));
    case VT_G2: return get_g2(r, reinterpret_cast<G2Aff*>(v->raw));
    case VT_FR: return get_fr(r, reinterpret_cast<Fr*>(v->raw));
  }
  return r.ok = false;
}
// IdentityOutput<T>(Vec<T>): u64 length (must be 1 here) then the element (identity/mod.rs:33-62)
static bool get_identity_out(Reader& r, int t, Val* v) {
  uint64_t len;
  if (!get_u64_le(r, &len) || len != 1) return r.ok = false;
  return get_val(r, t, v);
}
static bool val_eq(const Val& a, const Val& b) { return a.t == b.t && memcmp(a.raw, b.raw, vt_size(a.t)) == 0; }
static Val val_fr(const Fr& f) {
  Val v;
  v.t = VT_FR;
  memset(v.raw, 0, sizeof(v.raw));
  memcpy(v.raw, f.v, 32);
  return v;
}

// ------------------------------------------------------------------------------------------------
// subgroup membership of everything the readers decoded (ark-ec: is_in_correct_subgroup_assuming_on_curve;
// PairingOutput::check).  G1 / G2: serde::in_prime_subgroup (serde.cuh, shared with the point decoders of
// deserialize.cu); GT: k_gt_check6 (pairing6.cu).
// ------------------------------------------------------------------------------------------------
template <class F>
__global__ void __launch_bounds__(64) k_subgroup_check(const Aff<F>* __restrict__ pts, uint32_t n, uint32_t* __restrict__ bad,
                                                       uint32_t flag) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (!serde::in_prime_subgroup(pts[i])) atomicOr(bad, flag);
}

// *bad_mask: bit 0 = a G1 element, bit 1 = a G2 element, bit 2 = a GT element outside its prime-order subgroup
static int validate_subgroups(ripp_ctx* ctx, std::initializer_list<Reader*> readers, uint32_t* bad_mask) {
  std::vector<G1Aff> g1;
  std::vector<G2Aff> g2;
  std::vector<Fq12> gt;
  for (Reader* r : readers) {
    g1.insert(g1.end(), r->g1s.begin(), r->g1s.end());
    g2.insert(g2.end(), r->g2s.begin(), r->g2s.end());
    gt.insert(gt.end(), r->gts.begin(), r->gts.end());
  }
  *bad_mask = 0;
  if (g1.empty() && g2.empty() && gt.empty()) return RIPP_OK;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t o_g2 = up(g1.size() * 96), o_gt = o_g2 + up(g2.size() * 192), o_flag = o_gt + up(gt.size() * 576);
  void* d;
  OK(scratch(ctx, 21, o_flag + 256, &d));
  char* D = (char*)d;
  cudaStream_t st = ctx->stream;
  uint32_t* flag = (uint32_t*)(D + o_flag);
  CU(cudaMemsetAsync(flag, 0, 4, st));
  if (!g1.empty()) {
    CU(cudaMemcpyAsync(D, g1.data(), g1.size() * 96, cudaMemcpyHostToDevice, st));
    k_subgroup_check<Fq><<<(unsigned)((g1.size() + 63) / 64), 64, 0, st>>>((const G1Aff*)D, (uint32_t)g1.size(), flag, 1u);
    LAUNCHED(ctx);
  }
  if (!g2.empty()) {
    CU(cudaMemcpyAsync(D + o_g2, g2.data(), g2.size() * 192, cudaMemcpyHostToDevice, st));
    k_subgroup_check<Fq2><<<(unsigned)((g2.size() + 63) / 64), 64, 0, st>>>((const G2Aff*)(D + o_g2), (uint32_t)g2.size(), flag, 2u);
    LAUNCHED(ctx);
  }
  if (!gt.empty()) {
    CU(cudaMemcpyAsync(D + o_gt, gt.data(), gt.size() * 576, cudaMemcpyHostToDevice, st));
    OK(ripp_gt_check_l6(ctx, D + o_gt, gt.size(), flag, 4u));
  }
  CU(cudaMemcpyAsync(bad_mask, flag, 4, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return RIPP_OK;
}
static int subgroup_error(uint32_t mask) {
  return fail(RIPP_ERR_ARG, std::string("proof element outside the prime-order subgroup (ark-serialize would reject: InvalidData):") +
                                (mask & 1 ? " G1" : "") + (mask & 2 ? " G2" : "") + (mask & 4 ? " GT" : ""));
}

// ------------------------------------------------------------------------------------------------
// parsed proofs
// ------------------------------------------------------------------------------------------------
struct ComTypes {
  int l, r, t;  // LMC::Output, RMC::Output, element of IPC::Output
};
static ComTypes com_types(const GipaSpec& sp) {
  return ComTypes{ip_out_type(sp.a, sp.v), sp.w == VT_NONE ? VT_FR : ip_out_type(sp.w, sp.b), ip_out_type(sp.a, sp.b)};
}
struct GipaProofP {
  std::vector<std::vector<Val>> steps;  // stored order (last round first), 6 values each
  Val a0, b0;                           // r_base
};
static bool parse_gipa_proof(Reader& r, const GipaSpec& sp, GipaProofP* out) {
  ComTypes ct = com_types(sp);
  uint64_t k;
  if (!get_u64_le(r, &k) || k > 64) return r.ok = false;
  out->steps.assign(k, std::vector<Val>(6));
  for (uint64_t s = 0; s < k; s++)
    for (int h = 0; h < 2; h++) {
      Val* c = &out->steps[s][3 * h];
      if (!get_val(r, ct.l, &c[0]) || !get_val(r, ct.r, &c[1]) || !get_identity_out(r, ct.t, &c[2])) return false;
    }
  return get_val(r, sp.a, &out->a0) && get_val(r, sp.b, &out->b0);
}

// gipa.rs:322-363 challenges only: transcript in the reference's (reversed) order, element 0 = last round's c
static void recursive_challenges(const GipaProofP& pf, std::vector<Fr>* transcript, std::vector<Fr>* c_round,
                                 std::vector<Fr>* cinv_round) {
  size_t k = pf.steps.size();
  c_round->clear();
  cinv_round->clear();
  Fr prev = Fr::zero();
  for (size_t s = k; s-- > 0;) {  // proof.r_commitment_steps.iter().rev()
    Fr c, ci;
    gipa_challenge(prev, pf.steps[s].data(), &c, &ci);
    c_round->push_back(c);
    cinv_round->push_back(ci);
    prev = c;
  }
  transcript->assign(c_round->rbegin(), c_round->rend());
}

// sum_i scalars[i] * elems[i] in the group of type t (GT written additively, as PairingOutput is)
static int combine(ripp_ctx* ctx, int t, const std::vector<Val>& elems, const std::vector<Fr>& sc, Val* out) {
  out->t = t;
  memset(out->raw, 0, sizeof(out->raw));
  size_t n = elems.size();
  if (t == VT_FR) {
    Fr acc = Fr::zero();
    for (size_t i = 0; i < n; i++) acc = acc + *reinterpret_cast<const Fr*>(elems[i].raw) * sc[i];
    memcpy(out->raw, acc.v, 32);
    return RIPP_OK;
  }
  size_t es = vt_size(t);
  std::vector<uint8_t> host(n * es);
  for (size_t i = 0; i < n; i++) memcpy(&host[i * es], elems[i].raw, es);
  void* d;
  size_t off_sc = (n * es + 255) & ~(size_t)255, off_out = off_sc + ((n * 32 + 255) & ~(size_t)255);
  OK(scratch(ctx, 19, off_out + 1024, &d));
  char* D = (char*)d;
  CU(cudaMemcpyAsync(D, host.data(), n * es, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(D + off_sc, sc.data(), n * 32, cudaMemcpyHostToDevice, ctx->stream));
  if (t == VT_GT)
    OK(ripp_gt_multiexp_l6(ctx, D, D + off_sc, n, D + off_out));
  else if (t == VT_G1)
    OK(ripp_msm_g1_dev(ctx, D, D + off_sc, n, D + off_out));
  else
    OK(ripp_msm_g2_dev(ctx, D, D + off_sc, n, D + off_out));
  CU(cudaMemcpyAsync(out->raw, D + off_out, es, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

// base commitments of gipa.rs:355-357 after all rounds: com + sum_k (c_k com_1[k] + c_k^-1 com_2[k]), per component
static int fold_commitments(ripp_ctx* ctx, const GipaProofP& pf, const std::vector<Fr>& c_round,
                            const std::vector<Fr>& cinv_round, const Val com[3], Val base[3]) {
  size_t k = pf.steps.size();
  for (int j = 0; j < 3; j++) {
    std::vector<Val> el;
    std::vector<Fr> sc;
    el.push_back(com[j]);
    sc.push_back(Fr::one());
    for (size_t rd = 0; rd < k; rd++) {
      const std::vector<Val>& st = pf.steps[k - 1 - rd];
      el.push_back(st[j]);
      sc.push_back(c_round[rd]);
      el.push_back(st[3 + j]);
      sc.push_back(cinv_round[rd]);
    }
    OK(combine(ctx, com[j].t, el, sc, &base[j]));
  }
  return RIPP_OK;
}

// inner products of length-1 vectors held on the host (the base-case checks); result on the host
static int ip_single(ripp_ctx* ctx, int k, const Val* xs, const Val* ys, Val* out) {
  void* d;
  OK(scratch(ctx, 19, 2 * 8 * 576 + 1024, &d));
  char* D = (char*)d;
  Slice sx[8], sy[8];
  for (int i = 0; i < k; i++) {
    sx[i] = Slice{xs[i].t, D + 576 * (2 * i)};
    sy[i] = Slice{ys[i].t, D + 576 * (2 * i + 1)};
    if (xs[i].t != VT_NONE) CU(cudaMemcpyAsync(D + 576 * (2 * i), xs[i].raw, vt_size(xs[i].t), cudaMemcpyHostToDevice, ctx->stream));
    if (ys[i].t != VT_NONE) CU(cudaMemcpyAsync(D + 576 * (2 * i + 1), ys[i].raw, vt_size(ys[i].t), cudaMemcpyHostToDevice, ctx->stream));
  }
  return eval_products(ctx, k, sx, sy, 1, out);
}
static Val val_none() {
  Val v;
  v.t = VT_NONE;
  memset(v.raw, 0, sizeof(v.raw));
  return v;
}

// gipa.rs:401-415 with explicit base keys: LMC::verify([ck_a],[a0],com_a) && RMC::verify([ck_b],[b0],com_b)
// && IPC::verify(ck_t,[IP(a0,b0)],com_t).  b_override replaces b0 in the inner product (SSM final scalar).
static int verify_base(ripp_ctx* ctx, const GipaSpec& sp, const Val& ck_a, const Val* ck_b, const Val& a0, const Val& b0,
                       const Val base[3], bool check_rmc, bool* okp) {
  Val xs[3] = {a0, ck_b ? *ck_b : val_none(), a0};
  Val ys[3] = {ck_a, b0, b0};
  Val res[3];
  if (!check_rmc) {  // 2 products: LMC and the inner product
    xs[1] = a0;
    ys[1] = b0;
    OK(ip_single(ctx, 2, xs, ys, res));
    *okp = val_eq(res[0], base[0]) && val_eq(res[1], base[2]);
    return RIPP_OK;
  }
  (void)sp;
  OK(ip_single(ctx, 3, xs, ys, res));
  *okp = val_eq(res[0], base[0]) && val_eq(res[1], base[1]) && val_eq(res[2], base[2]);
  return RIPP_OK;
}

static bool parse_coms(Reader& r, const GipaSpec& sp, bool ssm, Val com[3]) {
  ComTypes ct = com_types(sp);
  if (!get_val(r, ct.l, &com[0])) return false;
  if (ssm)
    com[1] = val_fr(Fr::zero());
  else if (!get_val(r, ct.r, &com[1]))
    return false;
  return get_identity_out(r, ct.t, &com[2]);
}

// structured_scalar_message.rs:107-113 / :314-321: prod_j (1 + x_j^-1 b^(2^j)) over the (reversed) transcript
static Fr ssm_final_scalar(const std::vector<Fr>& transcript, const Fr& scalar_b) {
  Fr power = scalar_b, prod = Fr::one();
  for (size_t i = 0; i < transcript.size(); i++) {
    prod = prod * (Fr::one() + transcript[i].inv() * power);
    power = power * power;
  }
  return prod;
}

// ------------------------------------------------------------------------------------------------
// GIPA::verify (gipa.rs:135-160) and GIPAWithSSM::verify_with_structured_scalar_message (:86-127)
// ------------------------------------------------------------------------------------------------
// gipa.rs:365-399: exponents of the final keys; ck_a gets products of c^-1, ck_b products of c
static void final_key_exponents(const std::vector<Fr>& transcript, std::vector<Fr>* ea, std::vector<Fr>* eb) {
  ea->assign(1, Fr::one());
  eb->assign(1, Fr::one());
  for (size_t i = 0; i < transcript.size(); i++) {
    Fr c = transcript[i], ci = c.inv();
    size_t cur = (size_t)1 << i;
    for (size_t j = 0; j < cur; j++) {
      ea->push_back((*ea)[j] * ci);
      eb->push_back((*eb)[j] * c);
    }
  }
}
static int msm_typed(ripp_ctx* ctx, int t, const void* bases_dev, const std::vector<Fr>& sc, Val* out) {
  out->t = t;
  memset(out->raw, 0, sizeof(out->raw));
  void* d;
  size_t n = sc.size();
  OK(scratch(ctx, 19, n * 32 + 1024, &d));
  char* D = (char*)d;
  char* res = D + ((n * 32 + 255) & ~(size_t)255);
  CU(cudaMemcpyAsync(D, sc.data(), n * 32, cudaMemcpyHostToDevice, ctx->stream));
  if (t == VT_G1)
    OK(ripp_msm_g1_dev(ctx, bases_dev, D, n, res));
  else
    OK(ripp_msm_g2_dev(ctx, bases_dev, D, n, res));
  CU(cudaMemcpyAsync(out->raw, res, vt_size(t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

extern "C" int ripp_gipa_verify_dev(ripp_ctx* ctx, int kind, const void* v_dev, const void* w_dev, size_t n,
                                    const uint8_t* com, size_t com_len, const void* scalar_b, const uint8_t* proof,
                                    size_t proof_len, int* accept) {
  GipaSpec sp;
  if (!ctx || !accept || !gipa_spec(kind, &sp)) return fail(RIPP_ERR_ARG, "bad context, GIPA kind or output pointer");
  *accept = 0;
  bool ssm = sp.w == VT_NONE;
  if (!v_dev || (!ssm && !w_dev) || (ssm && !scalar_b)) return fail(RIPP_ERR_ARG, "null argument");
  // gipa.rs:140-146
  if (n == 0 || (n & (n - 1)))
    return fail(RIPP_ERR_NOT_POW2, "left length, right length: " + std::to_string(n) + ", " + std::to_string(n));
  CU(cudaSetDevice(ctx->device));
  Reader rc(com, com_len), rp(proof, proof_len);
  Val cm[3];
  GipaProofP pf;
  if (!parse_coms(rc, sp, ssm, cm) || !rc.done()) return fail(RIPP_ERR_ARG, "malformed commitment bytes");
  if (!parse_gipa_proof(rp, sp, &pf) || !rp.done()) return fail(RIPP_ERR_ARG, "malformed GIPA proof bytes");
  uint32_t bad = 0;
  OK(validate_subgroups(ctx, {&rc, &rp}, &bad));
  if (bad) return subgroup_error(bad);
  if (((size_t)1 << pf.steps.size()) != n) return RIPP_OK;  // transcript length does not match the keys: reject
  std::vector<Fr> transcript, c_round, cinv_round;
  recursive_challenges(pf, &transcript, &c_round, &cinv_round);
  Val base[3];
  OK(fold_commitments(ctx, pf, c_round, cinv_round, cm, base));
  std::vector<Fr> ea, eb;
  final_key_exponents(transcript, &ea, &eb);
  Val ck_a, ck_b;
  OK(msm_typed(ctx, sp.v, v_dev, ea, &ck_a));
  if (!ssm) OK(msm_typed(ctx, sp.w, w_dev, eb, &ck_b));
  bool ok = false;
  if (!ssm) {
    OK(verify_base(ctx, sp, ck_a, &ck_b, pf.a0, pf.b0, base, true, &ok));
  } else {
    // :95-105 gipa_valid: the placeholder commitment to r_base.1 is Fr::zero() and must equal the folded com_b
    bool ok1 = false, ok2 = false;
    OK(verify_base(ctx, sp, ck_a, nullptr, pf.a0, pf.b0, base, false, &ok1));
    ok1 = ok1 && val_eq(base[1], val_fr(Fr::zero()));
    // :107-125 base_valid with b_base recomputed from scalar_b
    Fr sb;
    memcpy(sb.v, scalar_b, 32);
    Val bb = val_fr(ssm_final_scalar(transcript, sb));
    OK(verify_base(ctx, sp, ck_a, nullptr, pf.a0, bb, base, false, &ok2));
    ok = ok1 && ok2;
  }
  *accept = ok ? 1 : 0;
  return RIPP_OK;
}

// ------------------------------------------------------------------------------------------------
// TIPA (tipa/mod.rs:242-301) and TIPA with structured scalar message (structured_scalar_message.rs:270-331)
// ------------------------------------------------------------------------------------------------
struct VerifierSRS {  // tipa/mod.rs:88-94, host, Montgomery affine: g | h | g_beta | h_alpha
  G1Aff g;
  G2Aff h;
  G1Aff g_beta;
  G2Aff h_alpha;
};
static VerifierSRS load_vsrs(const void* p) {
  VerifierSRS v;
  const char* c = (const char*)p;
  memcpy(&v.g, c, 96);
  memcpy(&v.h, c + 96, 192);
  memcpy(&v.g_beta, c + 288, 96);
  memcpy(&v.h_alpha, c + 384, 192);
  return v;
}
// tipa/mod.rs:393-405
static Fr poly_eval_product_form(const std::vector<Fr>& transcript, const Fr& z, const Fr& r_shift) {
  Fr power = z * z * r_shift, prod = Fr::one();
  for (size_t i = 0; i < transcript.size(); i++) {
    prod = prod * (Fr::one() + transcript[i] * power);
    power = power * power;
  }
  return prod;
}

// Both KZG checks of tipa/mod.rs:340-370 in one pairing batch.  With `g1_too == false` only the G2 opening.
//   e(g, ck_a - h f_a(z)) == e(g_beta - g z, pi_a);   e(ck_b - g f_b(z), h) == e(pi_b, h_alpha - h z)
static int kzg_checks(ripp_ctx* ctx, const VerifierSRS& vs, const G2Aff& ck_a, const G2Aff& pi_a, const Fr& eval_a,
                      const G1Aff* ck_b, const G1Aff* pi_b, const Fr& eval_b, const Fr& z, bool* okp) {
  void* d;
  OK(scratch(ctx, 19, 64 * 1024, &d));
  char* D = (char*)d;
  // staging: G1 slots of 96 B from 0, G2 slots of 192 B from 4096
  auto G1s = [&](int i) { return D + 96 * i; };
  auto G2s = [&](int i) { return D + 4096 + 192 * i; };
  cudaStream_t st = ctx->stream;
  const bool two = ck_b != nullptr;
  CU(cudaMemcpyAsync(G1s(0), &vs.g, 96, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(G1s(1), &vs.g_beta, 96, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(G2s(0), &vs.h, 192, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(G2s(1), &vs.h_alpha, 192, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(G2s(2), &ck_a, 192, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(G2s(3), &pi_a, 192, cudaMemcpyHostToDevice, st));
  if (two) {
    CU(cudaMemcpyAsync(G1s(2), ck_b, 96, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(G1s(3), pi_b, 96, cudaMemcpyHostToDevice, st));
  }
  Fr m_eval_a = -eval_a, m_eval_b = -eval_b, m_z = -z;
  // out = hi * c + lo with n = 1: the fold kernels are the point "a - s b" primitive
  OK(ripp_g2_fold_dev(ctx, G2s(0), G2s(2), m_eval_a.v, 1, G2s(4)));  // ck_a - h f_a(z)
  OK(ripp_g1_fold_dev(ctx, G1s(0), G1s(1), m_z.v, 1, G1s(4)));       // g_beta - g z
  if (two) {
    OK(ripp_g1_fold_dev(ctx, G1s(0), G1s(2), m_eval_b.v, 1, G1s(5)));  // ck_b - g f_b(z)
    OK(ripp_g2_fold_dev(ctx, G2s(0), G2s(1), m_z.v, 1, G2s(5)));       // h_alpha - h z
  }
  const void* g1[4] = {G1s(0), G1s(4), G1s(5), G1s(3)};
  const void* g2[4] = {G2s(4), G2s(3), G2s(0), G2s(5)};
  char* res = D + 16384;
  OK(ripp_pairing_batch_internal(ctx, two ? 4 : 2, g1, g2, 1, res));
  Fq12 out[4];
  CU(cudaMemcpyAsync(out, res, (two ? 4 : 2) * 576, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  *okp = memcmp(&out[0], &out[1], 576) == 0 && (!two || memcmp(&out[2], &out[3], 576) == 0);
  return RIPP_OK;
}

// com: com_a, com_b, com_t (non-SSM) / com_a, com_t (SSM).  shift: r_shift (non-SSM) / scalar_b (SSM).
static int tipa_verify_parsed(ripp_ctx* ctx, const GipaSpec& sp, const VerifierSRS& vs, const Val cm_in[3], const Fr& shift,
                              const GipaProofP& pf, const Val& ck_a_final, const Val* ck_b_final, const G2Aff& pi_a,
                              const G1Aff* pi_b, bool* okp) {
  const bool ssm = sp.w == VT_NONE;
  *okp = false;
  if (pf.steps.empty()) return RIPP_OK;  // transcript.first().unwrap() would panic: reject
  std::vector<Fr> transcript, c_round, cinv_round;
  recursive_challenges(pf, &transcript, &c_round, &cinv_round);
  Val cm[3] = {cm_in[0], cm_in[1], cm_in[2]};
  if (ssm) cm[1] = val_fr(shift);  // structured_scalar_message.rs:277-280 passes scalar_b as com_b (result unused)
  Val base[3];
  OK(fold_commitments(ctx, pf, c_round, cinv_round, cm, base));
  std::vector<Fr> tinv(transcript.size());
  for (size_t i = 0; i < tinv.size(); i++) tinv[i] = transcript[i].inv();
  // KZG challenge point (tipa/mod.rs:256-271 / structured_scalar_message.rs:288-301)
  Bytes parts;
  put_fr(parts, transcript[0]);
  put_val(parts, ck_a_final);
  if (!ssm) put_val(parts, *ck_b_final);
  Fr z = challenge_from_random_bytes(parts);
  bool kzg_ok = false;
  Fr shift_a = ssm ? Fr::one() : shift.inv();
  Fr eval_a = poly_eval_product_form(tinv, z, shift_a);
  Fr eval_b = ssm ? Fr::zero() : poly_eval_product_form(transcript, z, Fr::one());
  OK(kzg_checks(ctx, vs, *reinterpret_cast<const G2Aff*>(ck_a_final.raw), pi_a, eval_a,
                ssm ? nullptr : reinterpret_cast<const G1Aff*>(ck_b_final->raw), pi_b, eval_b, z, &kzg_ok));
  bool base_ok = false;
  if (!ssm) {
    OK(verify_base(ctx, sp, ck_a_final, ck_b_final, pf.a0, pf.b0, base, true, &base_ok));
  } else {
    Val bb = val_fr(ssm_final_scalar(transcript, shift));
    OK(verify_base(ctx, sp, ck_a_final, nullptr, pf.a0, bb, base, false, &base_ok));
  }
  *okp = kzg_ok && base_ok;
  return RIPP_OK;
}

struct TipaProofP {
  GipaProofP gipa;
  Val ck_a, ck_b;
  G2Aff pi_a;
  G1Aff pi_b;
};
static bool parse_tipa_proof(Reader& r, const GipaSpec& sp, TipaProofP* out) {
  if (!parse_gipa_proof(r, sp, &out->gipa)) return false;
  if (!get_val(r, VT_G2, &out->ck_a)) return false;
  if (sp.w != VT_NONE) {
    if (!get_val(r, VT_G1, &out->ck_b)) return false;
    return get_g2(r, &out->pi_a) && get_g1(r, &out->pi_b);
  }
  return get_g2(r, &out->pi_a);
}

extern "C" int ripp_tipa_verify(ripp_ctx* ctx, int kind, const void* vsrs, const uint8_t* com, size_t com_len,
                                const void* shift, const uint8_t* proof, size_t proof_len, int* accept) {
  GipaSpec sp;
  if (!ctx || !accept || !gipa_spec(kind, &sp)) return fail(RIPP_ERR_ARG, "bad context, GIPA kind or output pointer");
  *accept = 0;
  if (sp.v != VT_G2 || (sp.w != VT_G1 && sp.w != VT_NONE)) return fail(RIPP_ERR_ARG, "TIPA needs keys in (G2, G1)");
  bool ssm = sp.w == VT_NONE;
  if (!vsrs || (ssm && !shift)) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  VerifierSRS vs = load_vsrs(vsrs);
  Fr sh = Fr::one();
  if (shift) memcpy(sh.v, shift, 32);
  Reader rc(com, com_len), rp(proof, proof_len);
  Val cm[3];
  TipaProofP tp;
  if (!parse_coms(rc, sp, ssm, cm) || !rc.done()) return fail(RIPP_ERR_ARG, "malformed commitment bytes");
  if (!parse_tipa_proof(rp, sp, &tp) || !rp.done()) return fail(RIPP_ERR_ARG, "malformed TIPA proof bytes");
  uint32_t bad = 0;
  OK(validate_subgroups(ctx, {&rc, &rp}, &bad));
  if (bad) return subgroup_error(bad);
  bool ok = false;
  OK(tipa_verify_parsed(ctx, sp, vs, cm, sh, tp.gipa, tp.ck_a, ssm ? nullptr : &tp.ck_b, tp.pi_a, ssm ? nullptr : &tp.pi_b, &ok));
  *accept = ok ? 1 : 0;
  return RIPP_OK;
}

// ------------------------------------------------------------------------------------------------
// verify_aggregate_proof (applications/groth16_aggregation.rs:162-231)
// ------------------------------------------------------------------------------------------------
// ip[j] = sum_i inputs[i * m + j] * r^i  (the per-input ScalarInnerProduct of :209-217), one block per column
__global__ void __launch_bounds__(128) k_input_column_ip(const Fr* __restrict__ inputs, const Fr* __restrict__ r_pow, size_t n,
                                                         int m, Fr* __restrict__ out) {
  __shared__ Fr part[128];
  const int j = blockIdx.x;
  Fr acc = Fr::zero();
  for (size_t i = threadIdx.x; i < n; i += blockDim.x) acc = acc + inputs[i * m + j] * r_pow[i];
  part[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 64; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) part[threadIdx.x] = part[threadIdx.x] + part[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[j] = part[0];
}

extern "C" int ripp_tipp_verify_aggregate(ripp_ctx* ctx, const void* vsrs, const void* vk, size_t m,
                                          const void* public_inputs, size_t n, const uint8_t* proof, size_t proof_len,
                                          int* accept) {
  if (!ctx || !accept || !vsrs || !vk || !public_inputs || !proof) return fail(RIPP_ERR_ARG, "null argument");
  *accept = 0;
  if (n == 0 || m == 0 || m > 1024) return fail(RIPP_ERR_ARG, "need n >= 1 proofs and 1..1024 public inputs per proof");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  VerifierSRS vs = load_vsrs(vsrs);
  GipaSpec sp_ab, sp_c;
  gipa_spec(RIPP_GIPA_PAIRING, &sp_ab);
  gipa_spec(RIPP_GIPA_MULTIEXP_SSM, &sp_c);
  // AggregateProof { com_a, com_b, com_c, ip_ab, agg_c, tipa_proof_ab, tipa_proof_c } (:58-66)
  Reader rp(proof, proof_len);
  Val com_a, com_b, com_c, ip_ab, agg_c;
  TipaProofP pab, pc;
  if (!get_val(rp, VT_GT, &com_a) || !get_val(rp, VT_GT, &com_b) || !get_val(rp, VT_GT, &com_c) ||
      !get_val(rp, VT_GT, &ip_ab) || !get_val(rp, VT_G1, &agg_c) || !parse_tipa_proof(rp, sp_ab, &pab) ||
      !parse_tipa_proof(rp, sp_c, &pc) || !rp.done())
    return fail(RIPP_ERR_ARG, "malformed AggregateProof bytes");
  uint32_t bad = 0;
  OK(validate_subgroups(ctx, {&rp}, &bad));
  if (bad) return subgroup_error(bad);
  // :174-186 r
  Bytes parts;
  put_val(parts, com_a);
  put_val(parts, com_b);
  put_val(parts, com_c);
  Fr r = challenge_from_random_bytes(parts);
  // :189-206 the two TIPA proofs
  bool ok_ab = false, ok_c = false;
  {
    Val cm[3] = {com_a, com_b, ip_ab};
    OK(tipa_verify_parsed(ctx, sp_ab, vs, cm, r, pab.gipa, pab.ck_a, &pab.ck_b, pab.pi_a, &pab.pi_b, &ok_ab));
  }
  {
    Val cm[3] = {com_c, val_fr(Fr::zero()), agg_c};
    OK(tipa_verify_parsed(ctx, sp_c, vs, cm, r, pc.gipa, pc.ck_a, nullptr, pc.pi_a, nullptr, &ok_c));
  }
  // :210-212 r_sum = (r^n - 1) / (r - 1)
  Fr rn = Fr::one(), b = r;
  for (size_t e = n; e; e >>= 1) {
    if (e & 1) rn = rn * b;
    b = b * b;
  }
  Fr r_sum = (rn - Fr::one()) * (r - Fr::one()).inv();
  // vk: alpha_g1 | beta_g2 | gamma_g2 | delta_g2 | gamma_abc_g1[m + 1]
  const char* vkp = (const char*)vk;
  const size_t o_alpha = 0, o_beta = 96, o_gamma = 288, o_delta = 480, o_abc = 672;
  void* d;
  size_t in_bytes = n * m * 32, pw_bytes = n * 32;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t o_in = 0, o_pw = o_in + up(in_bytes), o_pwi = o_pw + up(pw_bytes), o_sc = o_pwi + up(pw_bytes),
         o_abcd = o_sc + up((m + 1) * 32), o_g1 = o_abcd + up((m + 1) * 96), o_g2 = o_g1 + up(3 * 96), o_res = o_g2 + up(3 * 192);
  OK(scratch(ctx, 20, o_res + 1024, &d));
  char* D = (char*)d;
  CU(cudaMemcpyAsync(D + o_in, public_inputs, in_bytes, cudaMemcpyHostToDevice, st));
  k_fr_powers<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(r, n, (Fr*)(D + o_pw), (Fr*)(D + o_pwi), r.inv());
  LAUNCHED(ctx);
  // :214-224 g_ic = gamma_abc[0] r_sum + sum_j gamma_abc[j + 1] <inputs[.][j], r_vec>
  CU(cudaMemcpyAsync(D + o_sc, r_sum.v, 32, cudaMemcpyHostToDevice, st));
  k_input_column_ip<<<(unsigned)m, 128, 0, st>>>((const Fr*)(D + o_in), (const Fr*)(D + o_pw), n, (int)m, (Fr*)(D + o_sc) + 1);
  LAUNCHED(ctx);
  CU(cudaMemcpyAsync(D + o_abcd, vkp + o_abc, (m + 1) * 96, cudaMemcpyHostToDevice, st));
  OK(ripp_msm_g1_dev(ctx, D + o_abcd, D + o_sc, m + 1, D + o_g1 + 96));  // slot 1: g_ic
  // :212 alpha_g1 * r_sum (slot 0); :226 agg_c (slot 2)
  CU(cudaMemcpyAsync(D + o_g1 + 192, vkp + o_alpha, 96, cudaMemcpyHostToDevice, st));  // staged in slot 2 first
  OK(ripp_g1_scale_dev(ctx, D + o_g1 + 192, D + o_sc, 1, D + o_g1));
  CU(cudaMemcpyAsync(D + o_g1 + 192, agg_c.raw, 96, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(D + o_g2, vkp + o_beta, 192, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(D + o_g2 + 192, vkp + o_gamma, 192, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(D + o_g2 + 384, vkp + o_delta, 192, cudaMemcpyHostToDevice, st));
  // :228 ip_ab == p1 + p2 + p3: one three-pair product with a shared final exponentiation
  OK(ripp_pairing_ip_dev(ctx, D + o_g1, D + o_g2, 3, D + o_res));
  Val ppe;
  ppe.t = VT_GT;
  CU(cudaMemcpyAsync(ppe.raw, D + o_res, 576, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  bool ppe_ok = val_eq(ppe, ip_ab);
  *accept = (ok_ab && ok_c && ppe_ok) ? 1 : 0;
  return RIPP_OK;
}

// ------------------------------------------------------------------------------------------------
// SIPP::verify (sipp/src/lib.rs:109-180)
// ------------------------------------------------------------------------------------------------
extern "C" int ripp_sipp_verify(ripp_ctx* ctx, const void* a_aff, const void* b_aff, const void* r, size_t n,
                                const void* value_gt, const uint8_t* proof, size_t proof_len, int* accept) {
  if (!ctx || !accept || !a_aff || !b_aff || !r || !value_gt || !proof) return fail(RIPP_ERR_ARG, "null argument");
  *accept = 0;
  // lib.rs:117-123
  if (n < 2 || (n & (n - 1))) return fail(RIPP_ERR_NOT_POW2, "SIPP needs a power-of-two length >= 2");
  size_t k = 0;
  while (((size_t)1 << k) < n) k++;
  if (proof_len != k * 1152) return fail(RIPP_ERR_ARG, "proof must hold log2(n) pairs of GT elements");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
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
  // lib.rs:134-150: challenges from the proof elements
  Reader rp(proof, proof_len);
  std::vector<Val> el;
  std::vector<Fr> sc, xs, xinvs;
  Val v0;
  v0.t = VT_GT;
  memcpy(v0.raw, value_gt, 576);
  el.push_back(v0);
  sc.push_back(Fr::one());
  for (size_t j = 0; j < k; j++) {
    Val zl, zr;
    if (!get_val(rp, VT_GT, &zl) || !get_val(rp, VT_GT, &zr)) return fail(RIPP_ERR_ARG, "malformed SIPP proof bytes");
    rng.absorb(Bytes(proof + 1152 * j, proof + 1152 * (j + 1)));
    Fr x = rng.next_u128();
    if (x.is_zero()) return RIPP_OK;  // batch_inversion would leave 0; the honest prover never produces it
    Fr xi = x.inv();
    xs.push_back(x);
    xinvs.push_back(xi);
    el.push_back(zl);
    sc.push_back(x);
    el.push_back(zr);
    sc.push_back(xi);
  }
  uint32_t bad = 0;
  OK(validate_subgroups(ctx, {&rp}, &bad));
  if (bad) return subgroup_error(bad);
  // lib.rs:152-160 z' = value + sum (z_l x + z_r x^-1)
  Val zp;
  OK(combine(ctx, VT_GT, el, sc, &zp));
  // lib.rs:162-173 s_i = prod_{j : bit (k-1-j) of i set} x_j (times r_i), s_invs likewise with x^-1
  std::vector<Fr> s(n, Fr::one()), sinv(n, Fr::one());
  for (size_t j = 0; j < k; j++) {
    size_t bit = (size_t)1 << (k - 1 - j);
    for (size_t i = 0; i < n; i++)
      if (i & bit) {
        s[i] = s[i] * xs[j];
        sinv[i] = sinv[i] * xinvs[j];
      }
  }
  const Fr* rr = (const Fr*)r;
  for (size_t i = 0; i < n; i++) s[i] = s[i] * rr[i];
  // lib.rs:174-177 a' = MSM(a, s), b' = MSM(b, s_invs), accept = e(a', b') == z'
  void* d;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  size_t o_a = 0, o_b = up(n * 96), o_s = o_b + up(n * 192), o_si = o_s + up(n * 32), o_ap = o_si + up(n * 32), o_bp = o_ap + 256,
         o_res = o_bp + 256;
  OK(scratch(ctx, 20, o_res + 1024, &d));
  char* D = (char*)d;
  CU(cudaMemcpyAsync(D + o_a, a_aff, n * 96, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(D + o_b, b_aff, n * 192, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(D + o_s, s.data(), n * 32, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(D + o_si, sinv.data(), n * 32, cudaMemcpyHostToDevice, st));
  OK(ripp_msm_g1_dev(ctx, D + o_a, D + o_s, n, D + o_ap));
  OK(ripp_msm_g2_dev(ctx, D + o_b, D + o_si, n, D + o_bp));
  OK(ripp_pairing_ip_dev(ctx, D + o_ap, D + o_bp, 1, D + o_res));
  Val got;
  got.t = VT_GT;
  CU(cudaMemcpyAsync(got.raw, D + o_res, 576, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  *accept = val_eq(got, zp) ? 1 : 0;
  return RIPP_OK;
}

// prod_i g_i^(s_i) in GT (device pointers; scalars Fr in Montgomery form): the `PairingOutput * Fr` sums of the
// verifiers as a primitive.
extern "C" int ripp_gt_multiexp_dev(ripp_ctx* ctx, const void* gt_dev, const void* fr_dev, size_t n, void* gt_out_dev) {
  if (!ctx || !gt_out_dev || (n && (!gt_dev || !fr_dev))) return fail(RIPP_ERR_ARG, "null argument");
  return ripp_gt_multiexp_l6(ctx, gt_dev, fr_dev, n, gt_out_dev);
}
