// verify_aggregate_proof for many aggregates under one VerifierSRS and one VerifyingKey, one status per aggregate
// (include/ripp_b200.h "ripp_tipp_verify_aggregate_batch").  Part of the gipa.cu translation unit, after verify.cuh,
// whose decoding and Fiat-Shamir helpers it shares.
//
// The single verifier is a chain of small synchronised steps.  Here the host parses every aggregate and recomputes
// every Fiat-Shamir chain first; each check of verify_aggregate_proof then becomes a group identity of one of three
// kinds, and the identities of all K aggregates share a fixed set of launches:
//   GT folds (4 per aggregate)  com + sum_k (c_k com_1[k] + c_k^-1 com_2[k]) of com_a, com_b, ip_ab (AB proof) and
//                               com_c (C proof): one power launch over all of them, one segmented product tree;
//   a G1 identity               agg_c + sum_k (c_k L_k + c_k^-1 R_k) - b_ssm a0_c == O (the C proof's base check);
//   pairing equations           prod_{j < 3} e(P_j, Q_j) == target, every scalar moved to the G1 side by bilinearity:
//     AB KZG, G2 key    e(g, ck_a) e(-f_a(z) g, h) e(z g - g_beta, pi_a) == 1       (e(g, ck_a - f_a h) == e(g_beta - z g, pi_a))
//     AB KZG, G1 key    e(ck_b - f_b(z) g + z pi_b, h) e(-pi_b, h_alpha) == 1       (e(ck_b - f_b g, h) == e(pi_b, h_alpha - z h))
//     C KZG, G2 key     as the AB one, with the C proof's ck_a, pi_a, z, f_a
//     base checks       e(a0, ck_a), e(ck_b, b0), e(a0, b0) (AB), e(a0_c, ck_a_c) (C) == their GT fold
//     PPE               e(r_sum alpha, beta) e(g_ic, gamma) e(agg_c, delta) == ip_ab
// Every G1 point of the equations and of the G1 identity is a short sum of scalar multiples of known points: one G1
// scaling launch over all terms, three segmented sums (3 terms per equation pair, 2k + 2 per G1 identity, m + 1 per
// g_ic).  The equations run on the six-lane engine, one group per equation (ripp_pairing_checks_l6).
#pragma once
#include "verify.cuh"

// ip[k][j] = sum_i inputs[row0[k] + i][j] r_k^i (k_input_column_ip per aggregate): one block per (aggregate k, column j);
// thread t walks rows t, t + 128, ... with r_k^t, stepping by r_k^128.  Written to out[k * stride + j]; zero for an
// aggregate with live[k] == 0.
__global__ void __launch_bounds__(128) k_input_column_ip_batch(const Fr* __restrict__ inputs, const Fr* __restrict__ r,
                                                               const uint64_t* __restrict__ row0, const uint8_t* __restrict__ live,
                                                               int m, Fr* __restrict__ out, size_t stride) {
  __shared__ Fr part[128];
  const int j = blockIdx.y;
  const size_t k = blockIdx.x;
  Fr acc = Fr::zero();
  if (live[k]) {
    Fr pw = Fr::one(), step = r[k];
    for (int b = 0; b < 7; b++) {
      if ((threadIdx.x >> b) & 1) pw = pw * step;
      step = step * step;
    }
    for (uint64_t i = row0[k] + threadIdx.x; i < row0[k + 1]; i += 128) {
      acc = acc + inputs[i * m + j] * pw;
      pw = pw * step;
    }
  }
  part[threadIdx.x] = acc;
  __syncthreads();
  for (int s = 64; s > 0; s >>= 1) {
    if ((int)threadIdx.x < s) part[threadIdx.x] = part[threadIdx.x] + part[threadIdx.x + s];
    __syncthreads();
  }
  if (threadIdx.x == 0) out[k * stride + j] = part[0];
}

struct AggBatchItem {
  size_t n;
  Reader rd;
  AggregateProofP p;
  uint8_t status;
  // the Fiat-Shamir chain (host): round challenges of both proofs, KZG points and evaluations
  std::vector<Fr> c_ab, ci_ab, c_c, ci_c;
  Fr r, r_sum, z_ab, z_c, fa_ab, fb_ab, fa_c, b_ssm;
  AggBatchItem(const uint8_t* bytes, size_t len, size_t n_) : n(n_), rd(bytes, len), status(RIPP_AGG_OK) {}
};

// tipa_verify_parsed's challenges for both proofs of one aggregate (both have at least one round)
static void agg_fiat_shamir(AggBatchItem& a) {
  const AggregateProofP& p = a.p;
  a.r = aggregate_challenge(p.com_a, p.com_b, p.com_c);
  a.r_sum = aggregate_r_sum(a.r, a.n);
  std::vector<Fr> t, tinv;
  auto inverses = [&] {
    tinv.resize(t.size());
    for (size_t i = 0; i < t.size(); i++) tinv[i] = t[i].inv();
  };
  recursive_challenges(p.pab.gipa, &t, &a.c_ab, &a.ci_ab);
  inverses();
  {
    Bytes parts;
    put_fr(parts, t[0]);
    put_val(parts, p.pab.ck_a);
    put_val(parts, p.pab.ck_b);
    a.z_ab = challenge_from_random_bytes(parts);
  }
  a.fa_ab = poly_eval_product_form(tinv, a.z_ab, a.r.inv());
  a.fb_ab = poly_eval_product_form(t, a.z_ab, Fr::one());
  recursive_challenges(p.pc.gipa, &t, &a.c_c, &a.ci_c);
  inverses();
  {
    Bytes parts;
    put_fr(parts, t[0]);
    put_val(parts, p.pc.ck_a);
    a.z_c = challenge_from_random_bytes(parts);
  }
  a.fa_c = poly_eval_product_form(tinv, a.z_c, Fr::one());
  a.b_ssm = ssm_final_scalar(t, a.r);
}

static size_t up256(size_t x) { return (x + 255) & ~(size_t)255; }

// the elements one reader decoded and the word of the failure flags they set
struct SubgroupSrc {
  const Reader* rd;
  uint32_t owner;
};

// Subgroup checks of the elements of every source, one launch per group, a failure ORed into (*bad_h)[owner] (K words).
// host_work runs while the checks do; one synchronisation.
template <class Fn>
static int batch_subgroups(ripp_ctx* ctx, const std::vector<SubgroupSrc>& src, size_t K, Fn host_work, std::vector<uint32_t>* bad_h) {
  std::vector<G1Aff> g1;
  std::vector<G2Aff> g2;
  std::vector<Fq12> gt;
  std::vector<uint32_t> o1, o2, ot;
  for (const SubgroupSrc& s : src) {
    const Reader& r = *s.rd;
    g1.insert(g1.end(), r.g1s.begin(), r.g1s.end());
    g2.insert(g2.end(), r.g2s.begin(), r.g2s.end());
    gt.insert(gt.end(), r.gts.begin(), r.gts.end());
    o1.resize(g1.size(), s.owner);
    o2.resize(g2.size(), s.owner);
    ot.resize(gt.size(), s.owner);
  }
  const size_t o_g2 = up256(g1.size() * 96), o_gt = o_g2 + up256(g2.size() * 192),
               o_o1 = o_gt + up256(gt.size() * 576), o_o2 = o_o1 + up256(o1.size() * 4), o_ot = o_o2 + up256(o2.size() * 4),
               o_bad = o_ot + up256(ot.size() * 4);
  std::vector<uint8_t> H(o_bad);
  memcpy(H.data(), g1.data(), g1.size() * 96);
  memcpy(H.data() + o_g2, g2.data(), g2.size() * 192);
  memcpy(H.data() + o_gt, gt.data(), gt.size() * 576);
  memcpy(H.data() + o_o1, o1.data(), o1.size() * 4);
  memcpy(H.data() + o_o2, o2.data(), o2.size() * 4);
  memcpy(H.data() + o_ot, ot.data(), ot.size() * 4);
  void* d;
  OK(scratch(ctx, 38, o_bad + K * 4, &d));
  uint8_t* D = (uint8_t*)d;
  uint32_t* bad = (uint32_t*)(D + o_bad);
  cudaStream_t st = ctx->stream;
  CU(cudaMemcpyAsync(D, H.data(), o_bad, cudaMemcpyHostToDevice, st));
  CU(cudaMemsetAsync(bad, 0, K * 4, st));
  if (!g1.empty()) {
    k_subgroup_check<Fq><<<(unsigned)((g1.size() + 63) / 64), 64, 0, st>>>((const G1Aff*)D, (uint32_t)g1.size(), bad, 1u,
                                                                          (const uint32_t*)(D + o_o1));
    LAUNCHED(ctx);
  }
  if (!g2.empty()) {
    k_subgroup_check<Fq2><<<(unsigned)((g2.size() + 63) / 64), 64, 0, st>>>((const G2Aff*)(D + o_g2), (uint32_t)g2.size(), bad,
                                                                           2u, (const uint32_t*)(D + o_o2));
    LAUNCHED(ctx);
  }
  OK(ripp_gt_check_l6(ctx, D + o_gt, gt.size(), bad, 4u, (const uint32_t*)(D + o_ot)));
  host_work();
  bad_h->assign(K, 0);
  CU(cudaMemcpyAsync(bad_h->data(), bad, K * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return RIPP_OK;
}

// Subgroup checks of every decoded element of the aggregates with status OK, failures recorded per aggregate, and the
// host Fiat-Shamir work while they run.
static int agg_subgroups(ripp_ctx* ctx, std::vector<AggBatchItem>& it) {
  const size_t K = it.size();
  std::vector<SubgroupSrc> src;
  for (size_t k = 0; k < K; k++)
    if (it[k].status == RIPP_AGG_OK) src.push_back(SubgroupSrc{&it[k].rd, (uint32_t)k});
  std::vector<uint32_t> bad_h;
  OK(batch_subgroups(ctx, src, K, [&] {
    // tipa_verify_parsed rejects a proof without rounds (its transcript has no first element)
    for (AggBatchItem& a : it) {
      if (a.status != RIPP_AGG_OK) continue;
      if (a.p.pab.gipa.steps.empty() || a.p.pc.gipa.steps.empty())
        a.status = RIPP_AGG_REJECTED;
      else
        agg_fiat_shamir(a);
    }
  }, &bad_h));
  for (size_t k = 0; k < K; k++)
    if (bad_h[k] && it[k].status != RIPP_AGG_MALFORMED) it[k].status = RIPP_AGG_NOT_IN_SUBGROUP;
  return RIPP_OK;
}

extern "C" int ripp_tipp_verify_aggregate_batch(ripp_ctx* ctx, const void* vsrs, const void* vk, size_t m, size_t count,
                                                const size_t* n, const void* public_inputs, const uint8_t* proofs,
                                                size_t proofs_len, const size_t* proof_lens, uint8_t* status_out,
                                                size_t* n_accepted) {
  if (!ctx || !vsrs || !vk || !n_accepted) return fail(RIPP_ERR_ARG, "null argument");
  *n_accepted = 0;
  if (m == 0 || m > 1024) return fail(RIPP_ERR_ARG, "need 1..1024 public inputs per proof");
  if (count == 0) return RIPP_OK;
  if (!n || !public_inputs || !proofs || !proof_lens || !status_out) return fail(RIPP_ERR_ARG, "null argument");
  if (count > ((size_t)1 << 24)) return fail(RIPP_ERR_ARG, "more than 2^24 aggregates");
  size_t sum = 0, rows = 0;
  for (size_t k = 0; k < count; k++) {
    if (n[k] == 0) return fail(RIPP_ERR_ARG, "aggregate " + std::to_string(k) + " has n = 0 proofs");
    if (proof_lens[k] > proofs_len - sum)
      return fail(RIPP_ERR_ARG, "proof_lens add up to more than proofs_len = " + std::to_string(proofs_len));
    sum += proof_lens[k];
    rows += n[k];
  }
  if (sum != proofs_len)
    return fail(RIPP_ERR_ARG, "proof_lens add up to " + std::to_string(sum) + ", not proofs_len = " + std::to_string(proofs_len));
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const VerifierSRS vs = load_vsrs(vsrs);
  std::vector<AggBatchItem> it;
  it.reserve(count);
  for (size_t k = 0, off = 0; k < count; off += proof_lens[k], k++) {
    it.emplace_back(proofs + off, proof_lens[k], n[k]);
    if (!parse_aggregate_proof(it.back().rd, &it.back().p)) it.back().status = RIPP_AGG_MALFORMED;
  }
  OK(agg_subgroups(ctx, it));

  // ---- every check of the members still OK, in one set of launches ----
  const size_t K = count, E = 8 * K, M1 = m + 1;
  size_t LG = 1, LD = 1;  // longest GT fold, longest G1 identity
  bool any = false;
  for (const AggBatchItem& a : it) {
    if (a.status != RIPP_AGG_OK) continue;
    any = true;
    const size_t kab = a.p.pab.gipa.steps.size(), kc = a.p.pc.gipa.steps.size();
    LG = std::max(LG, 2 * std::max(kab, kc) + 1);
    LD = std::max(LD, 2 * kc + 2);
  }
  if (!any) {
    for (size_t k = 0; k < K; k++) status_out[k] = it[k].status;
    return RIPP_OK;
  }
  // G1 terms: [equation pairs: (j * E + e) * 3 + t | G1 identities: K x LD | g_ic: K x M1]
  const size_t o_D = 9 * E, o_ic = o_D + K * LD, nT = o_ic + K * M1;
  // host staging, uploaded in one copy; all-zero bytes are the identity (points) and zero (scalars)
  const size_t o_ts = up256(nT * 96), o_q = o_ts + up256(nT * 32), o_ge = o_q + up256(3 * E * 192),
               o_gs = o_ge + up256(4 * K * LG * 576), o_tg = o_gs + up256(4 * K * LG * 32), o_rk = o_tg + up256(E * 576),
               o_r0 = o_rk + up256(K * 32), o_lv = o_r0 + up256((K + 1) * 8), hbytes = o_lv + up256(K);
  std::vector<uint8_t> H(hbytes);
  G1Aff* TB = (G1Aff*)H.data();
  Fr* TS = (Fr*)(H.data() + o_ts);
  G2Aff* Q = (G2Aff*)(H.data() + o_q);
  Fq12* GE = (Fq12*)(H.data() + o_ge);
  Fr* GS = (Fr*)(H.data() + o_gs);
  Fq12* TG = (Fq12*)(H.data() + o_tg);
  Fr* RK = (Fr*)(H.data() + o_rk);
  uint64_t* R0 = (uint64_t*)(H.data() + o_r0);
  uint8_t* LV = H.data() + o_lv;
  const char* vkp = (const char*)vk;
  const G1Aff alpha = *(const G1Aff*)vkp;
  const G2Aff beta = *(const G2Aff*)(vkp + 96), gamma = *(const G2Aff*)(vkp + 288), delta = *(const G2Aff*)(vkp + 480);
  const Fr one = Fr::one(), m_one = -Fr::one();
  for (size_t i = 0; i < 4 * K * LG; i++) GE[i] = Fq12::one();
  for (size_t e = 4 * K; e < E; e++) TG[e] = Fq12::one();
  auto term = [&](size_t j, size_t e, int t, const G1Aff& b, const Fr& s) {
    TB[(j * E + e) * 3 + t] = b;
    TS[(j * E + e) * 3 + t] = s;
  };
  std::vector<Val> el;
  std::vector<Fr> sc;
  auto gt_fold = [&](size_t seg) {
    for (size_t i = 0; i < el.size(); i++) {
      memcpy(&GE[seg * LG + i], el[i].raw, 576);
      GS[seg * LG + i] = sc[i];
    }
  };
  R0[0] = 0;
  for (size_t k = 0; k < K; k++) {
    R0[k + 1] = R0[k] + n[k];
    const AggBatchItem& a = it[k];
    if (a.status != RIPP_AGG_OK) continue;
    LV[k] = 1;
    RK[k] = a.r;
    const AggregateProofP& p = a.p;
    const G1Aff &a0 = *(const G1Aff*)p.pab.gipa.a0.raw, &ck_b = *(const G1Aff*)p.pab.ck_b.raw, &a0_c = *(const G1Aff*)p.pc.gipa.a0.raw,
                &agg_c = *(const G1Aff*)p.agg_c.raw;
    const G2Aff &b0 = *(const G2Aff*)p.pab.gipa.b0.raw, &ck_a = *(const G2Aff*)p.pab.ck_a.raw, &ck_a_c = *(const G2Aff*)p.pc.ck_a.raw;
    // base checks against the folds (targets 0 .. 4K, written by the GT fold)
    size_t e = 4 * k;
    term(0, e, 0, a0, one);
    Q[e] = ck_a;
    term(0, e + 1, 0, ck_b, one);
    Q[e + 1] = b0;
    term(0, e + 2, 0, a0, one);
    Q[e + 2] = b0;
    term(0, e + 3, 0, a0_c, one);
    Q[e + 3] = ck_a_c;
    // PPE; pair 1's point g_ic comes from its own segmented sum
    e = 4 * K + k;
    term(0, e, 0, alpha, a.r_sum);
    Q[e] = beta;
    Q[E + e] = gamma;
    term(2, e, 0, agg_c, one);
    Q[2 * E + e] = delta;
    memcpy(&TG[e], p.ip_ab.raw, 576);
    // KZG openings of the final G2 keys (AB at 5K + k, C at 7K + k)
    auto kzg_g2 = [&](size_t q, const G2Aff& ck, const G2Aff& pi, const Fr& fa, const Fr& z) {
      term(0, q, 0, vs.g, one);
      Q[q] = ck;
      term(1, q, 0, vs.g, -fa);
      Q[E + q] = vs.h;
      term(2, q, 0, vs.g, z);
      term(2, q, 1, vs.g_beta, m_one);
      Q[2 * E + q] = pi;
    };
    kzg_g2(5 * K + k, ck_a, p.pab.pi_a, a.fa_ab, a.z_ab);
    kzg_g2(7 * K + k, ck_a_c, p.pc.pi_a, a.fa_c, a.z_c);
    // KZG opening of the final G1 key of the AB proof
    e = 6 * K + k;
    term(0, e, 0, ck_b, one);
    term(0, e, 1, vs.g, -a.fb_ab);
    term(0, e, 2, p.pab.pi_b, a.z_ab);
    Q[e] = vs.h;
    term(1, e, 0, p.pab.pi_b, m_one);
    Q[E + e] = vs.h_alpha;
    // the C proof's G1 identity: fold of agg_c minus b_ssm a0_c
    fold_terms(p.pc.gipa, a.c_c, a.ci_c, p.agg_c, 2, &el, &sc);
    for (size_t i = 0; i < el.size(); i++) {
      memcpy(&TB[o_D + k * LD + i], el[i].raw, 96);
      TS[o_D + k * LD + i] = sc[i];
    }
    TB[o_D + k * LD + el.size()] = a0_c;
    TS[o_D + k * LD + el.size()] = -a.b_ssm;
    // g_ic = r_sum IC_0 + sum_j ip_j IC_{j+1}; ip_j from k_input_column_ip_batch
    memcpy(&TB[o_ic + k * M1], vkp + 672, M1 * 96);
    TS[o_ic + k * M1] = a.r_sum;
    // GT folds: com_a, com_b, ip_ab of the AB proof, com_c of the C proof
    const Val com_ab[3] = {p.com_a, p.com_b, p.ip_ab};
    for (int j = 0; j < 3; j++) {
      fold_terms(p.pab.gipa, a.c_ab, a.ci_ab, com_ab[j], j, &el, &sc);
      gt_fold(4 * k + j);
    }
    fold_terms(p.pc.gipa, a.c_c, a.ci_c, p.com_c, 0, &el, &sc);
    gt_fold(4 * k + 3);
  }

  // device: [scaled terms | P (3 x E) | G1 identities (K) | Miller values (E) | verdicts (E) | public inputs]
  const size_t in_bytes = rows * m * 32, o_P = up256(nT * 96), o_id = o_P + up256(3 * E * 96), o_ml = o_id + up256(K * 96),
               o_ok = o_ml + up256(E * 576), o_in = o_ok + up256(E), dbytes = o_in + up256(in_bytes);
  void *hd, *dd;
  OK(scratch(ctx, 39, hbytes, &hd));
  OK(scratch(ctx, 40, dbytes, &dd));
  uint8_t *Dh = (uint8_t*)hd, *Dd = (uint8_t*)dd;
  const G1Aff* scaled = (const G1Aff*)Dd;
  G1Aff* P = (G1Aff*)(Dd + o_P);
  CU(cudaMemcpyAsync(Dh, H.data(), hbytes, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(Dd + o_in, public_inputs, in_bytes, cudaMemcpyHostToDevice, st));
  k_input_column_ip_batch<<<dim3((unsigned)K, (unsigned)m), 128, 0, st>>>((const Fr*)(Dd + o_in), (const Fr*)(Dh + o_rk),
                                                                         (const uint64_t*)(Dh + o_r0), Dh + o_lv, (int)m,
                                                                         (Fr*)(Dh + o_ts) + o_ic + 1, M1);
  LAUNCHED(ctx);
  OK(ripp_g1_scale_dev(ctx, Dh, Dh + o_ts, nT, Dd));
  OK(ripp_seg_sum_dev(ctx, 1, scaled, 3, (int)(3 * E), P));
  OK(ripp_seg_sum_dev(ctx, 1, scaled + o_D, LD, (int)K, Dd + o_id));
  OK(ripp_seg_sum_dev(ctx, 1, scaled + o_ic, M1, (int)K, P + E + 4 * K));
  OK(ripp_gt_multiexp_l6(ctx, Dh + o_ge, Dh + o_gs, LG, Dh + o_tg, (int)(4 * K)));
  OK(ripp_pairing_checks_l6(ctx, P, Dh + o_q, E, Dd + o_ml, Dh + o_tg, Dd + o_ok));
  std::vector<uint8_t> ok(E);
  std::vector<G1Aff> id(K);
  CU(cudaMemcpyAsync(ok.data(), Dd + o_ok, E, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(id.data(), Dd + o_id, K * 96, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  size_t acc = 0;
  for (size_t k = 0; k < K; k++) {
    AggBatchItem& a = it[k];
    if (a.status == RIPP_AGG_OK) {
      const bool eq = ok[4 * k] && ok[4 * k + 1] && ok[4 * k + 2] && ok[4 * k + 3] && ok[4 * K + k] && ok[5 * K + k] &&
                      ok[6 * K + k] && ok[7 * K + k];
      a.status = eq && id[k].is_inf() ? RIPP_AGG_OK : RIPP_AGG_REJECTED;
    }
    status_out[k] = a.status;
    acc += a.status == RIPP_AGG_OK;
  }
  *n_accepted = acc;
  return RIPP_OK;
}
