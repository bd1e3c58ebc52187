// ripp_pc_verify for many openings in one call, one status per opening (include/ripp_b200.h "ripp_pc_verify_batch").
// Part of the gipa.cu translation unit, after pc_batch.cuh: it shares the decoders and Fiat-Shamir helpers of
// verify.cuh, the subgroup checks and staging of verify_batch.cuh and the shape rules of poly_commit.cuh.
//
// The host parses every opening as ripp_pc_verify does and recomputes every transcript while the subgroup checks run.
// Every check of the single verifier is then an exact identity in a prime-order group (its elements have passed their
// subgroup checks), and the identities of all K openings share one fixed set of launches:
//   trusted (ripp_tipa_verify with MULTIEXP_SSM, then kzg_verify)
//     GT fold        com_gt + sum_r (c_r com_1[r] + c_r^-1 com_2[r])
//     G1 identity    fold of y_eval_comm - ssm(t, x) a0 == O
//     equations      e(g, ck) e(-f_a(z) g, h) e(z g - g_beta, pi) == 1                   (the final G2 key's opening)
//                    e(a0, ck) == GT fold                                                 (base check)
//                    e(y_eval_comm - eval g + y pi_kzg, h) e(-pi_kzg, h_alpha) == 1        (KZG opening at y)
//   transparent (two ripp_gipa_verify_dev)
//     second tier    log2 n rounds; GT fold == e(a0, ck2), ck2 = sum_i e2_i v_i; fold of the Fr placeholders == 0
//                    (host); fold of y_eval_comm - b0 a0 == O and fold of y_eval_comm - ssm(t2, x) a0 == O (both kept:
//                    with a0 = O and b0 != ssm the single verifier accepts, so b0 == ssm is not a check)
//     first tier     log2 m rounds; fold of y_eval_comm - a0 ck1 == O, ck1 = sum_i e1_i w_i; fold of the Fr
//                    placeholders == 0, fold of eval == a0 b0 == a0 ssm(t1, y) (host)
// Launches: the subgroup checks (sync); one staging upload; transparent: the final keys' exponents on the device
// (k_pc_key_exponents_seg) and two segmented MSMs over the shared keys, written straight into the staged slots; one G1
// scaling; two segmented sums; one GT multi-exponentiation over K segments; one pairing-check launch pair (sync).
#pragma once

// out[k 2^L + e] = factor_k prod_{bit j of e set} tinv[k L + j] (factor_k = 1 without `factor`): the exponents of
// count final commitment keys of 2^L elements (pc::key_exponent)
__global__ void k_pc_key_exponents_seg(const Fr* __restrict__ tinv, unsigned L, const Fr* __restrict__ factor, size_t count,
                                       Fr* __restrict__ out) {
  const size_t len = (size_t)1 << L, t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count * len) return;
  size_t k, e;
  pc::seg_split(t, len, &k, &e);
  out[t] = pc::key_exponent(tinv + k * L, e, factor ? factor[k] : Fr::one());
}

struct PcVerifyItem {
  uint8_t status = RIPP_AGG_OK;
  bool b_ok = false;  // the second stage decoded
  // stage A: trusted, the trailing y_eval_comm || kzg_proof; transparent, com || second-tier proof.
  // stage B: trusted, com || TIPA proof; transparent, y_eval_comm || eval || first-tier proof.
  Reader r[4] = {Reader(nullptr, 0), Reader(nullptr, 0), Reader(nullptr, 0), Reader(nullptr, 0)};
  Bytes ca, cb;       // the commitment bytes the readers decode
  Val com2[3], com1[3];
  GipaProofP p2, p1;  // second tier (trusted: the TIPA's GIPA), first tier
  TipaProofP tp;
  G1Aff ye, pik;      // trusted: y_eval_comm, kzg_proof
  std::vector<Fr> t2, c2, ci2, t1, c1, ci1;
  Fr z, fa, ssm2, ssm1;
};

static Fr fr_fold(const std::vector<Val>& el, const std::vector<Fr>& sc) {
  Fr acc = Fr::zero();
  for (size_t i = 0; i < el.size(); i++) acc = acc + *reinterpret_cast<const Fr*>(el[i].raw) * sc[i];
  return acc;
}

static size_t log2_pow2(size_t n) {
  size_t k = 0;
  while (((size_t)1 << k) < n) k++;
  return k;
}

// ripp_pc_verify's decoding of opening k into its two stages
static void pc_verify_parse(PcVerifyItem& a, bool trusted, size_t n, const Fq12& com_gt, const Fr& eval, const uint8_t* pf, size_t len) {
  GipaSpec s2, s1;
  gipa_spec(RIPP_GIPA_MULTIEXP_SSM, &s2);
  gipa_spec(RIPP_GIPA_SCALAR_SSM_G1, &s1);
  if (trusted) {
    if (len < 192) {
      a.status = RIPP_AGG_MALFORMED;
      return;
    }
    const uint8_t* ye = pf + len - 192;
    a.r[0] = Reader(ye, 192);
    if (!get_g1(a.r[0], &a.ye) || !get_g1(a.r[0], &a.pik) || !a.r[0].done()) {
      a.status = RIPP_AGG_MALFORMED;
      return;
    }
    put_gt(a.cb, com_gt);
    put_u64_le(a.cb, 1);
    a.cb.insert(a.cb.end(), ye, ye + 96);
    a.r[2] = Reader(a.cb.data(), a.cb.size());
    a.r[3] = Reader(pf, len - 192);
    a.b_ok = parse_coms(a.r[2], s2, true, a.com2) && a.r[2].done() && parse_tipa_proof(a.r[3], s2, &a.tp) && a.r[3].done();
    return;
  }
  const size_t s = transparent_second_len(n);
  if (len < s + 96) {
    a.status = RIPP_AGG_MALFORMED;
    return;
  }
  const uint8_t* ye = pf + s;
  put_gt(a.ca, com_gt);
  put_u64_le(a.ca, 1);
  a.ca.insert(a.ca.end(), ye, ye + 96);
  a.r[0] = Reader(a.ca.data(), a.ca.size());
  a.r[1] = Reader(pf, s);
  if (!parse_coms(a.r[0], s2, true, a.com2) || !a.r[0].done() || !parse_gipa_proof(a.r[1], s2, &a.p2) || !a.r[1].done()) {
    a.status = RIPP_AGG_MALFORMED;
    return;
  }
  a.cb.insert(a.cb.end(), ye, ye + 96);
  put_u64_le(a.cb, 1);
  put_fr(a.cb, eval);
  a.r[2] = Reader(a.cb.data(), a.cb.size());
  a.r[3] = Reader(ye + 96, len - s - 96);
  a.b_ok = parse_coms(a.r[2], s1, true, a.com1) && a.r[2].done() && parse_gipa_proof(a.r[3], s1, &a.p1) && a.r[3].done();
}

// the Fiat-Shamir chains of one decoded opening and its host checks (REJECTED where one fails)
static void pc_verify_host(PcVerifyItem& a, bool trusted, size_t L2, size_t L1, const Fr& x, const Fr& y) {
  std::vector<Val> el;
  std::vector<Fr> sc;
  if (trusted) {
    const GipaProofP& g = a.tp.gipa;
    if (g.steps.empty()) {  // tipa_verify_parsed: no first transcript element
      a.status = RIPP_AGG_REJECTED;
      return;
    }
    recursive_challenges(g, &a.t2, &a.c2, &a.ci2);
    std::vector<Fr> tinv(a.t2.size());
    for (size_t i = 0; i < tinv.size(); i++) tinv[i] = a.t2[i].inv();
    Bytes parts;
    put_fr(parts, a.t2[0]);
    put_val(parts, a.tp.ck_a);
    a.z = challenge_from_random_bytes(parts);
    a.fa = poly_eval_product_form(tinv, a.z, Fr::one());
    a.ssm2 = ssm_final_scalar(a.t2, x);
    return;
  }
  if (a.p2.steps.size() != L2 || a.p1.steps.size() != L1) {  // the transcript does not match the keys
    a.status = RIPP_AGG_REJECTED;
    return;
  }
  recursive_challenges(a.p2, &a.t2, &a.c2, &a.ci2);
  recursive_challenges(a.p1, &a.t1, &a.c1, &a.ci1);
  a.ssm2 = ssm_final_scalar(a.t2, x);
  a.ssm1 = ssm_final_scalar(a.t1, y);
  fold_terms(a.p2, a.c2, a.ci2, a.com2[1], 1, &el, &sc);
  bool ok = fr_fold(el, sc).is_zero();
  fold_terms(a.p1, a.c1, a.ci1, a.com1[1], 1, &el, &sc);
  ok = ok && fr_fold(el, sc).is_zero();
  fold_terms(a.p1, a.c1, a.ci1, a.com1[2], 2, &el, &sc);
  const Fr ev = fr_fold(el, sc), a0 = *(const Fr*)a.p1.a0.raw, b0 = *(const Fr*)a.p1.b0.raw;
  ok = ok && ev == a0 * b0 && ev == a0 * a.ssm1;
  if (!ok) a.status = RIPP_AGG_REJECTED;
}

extern "C" int ripp_pc_verify_batch(ripp_ctx* ctx, int kind, const void* vsrs, const void* first_tier_dev, size_t m,
                                    const void* second_tier_dev, size_t n, size_t count, const void* com_gts, const void* x_host,
                                    const void* y_host, const void* evals, const uint8_t* proofs, size_t proofs_len,
                                    const size_t* proof_lens, uint8_t* status_out, size_t* n_accepted) {
  if (!ctx || !n_accepted) return fail(RIPP_ERR_ARG, "null argument");
  *n_accepted = 0;
  if (kind != RIPP_PC_TRUSTED && kind != RIPP_PC_TRANSPARENT) return fail(RIPP_ERR_ARG, "bad polynomial-commitment kind");
  if (count == 0) return RIPP_OK;
  if (!com_gts || !x_host || !y_host || !evals || !proofs || !proof_lens || !status_out) return fail(RIPP_ERR_ARG, "null argument");
  const bool trusted = kind == RIPP_PC_TRUSTED;
  if (trusted && !vsrs) return fail(RIPP_ERR_ARG, "null argument: the trusted kind needs the VerifierSRS");
  if (!trusted) {
    if (!first_tier_dev || !second_tier_dev) return fail(RIPP_ERR_ARG, "null argument");
    OK(pc_shape(n, m, 0));
  }
  const size_t lim = (size_t)1 << 24;
  if (count > ((size_t)1 << 16) || (!trusted && (count > lim / n || count > lim / m)))
    return fail(RIPP_ERR_ARG, "polynomial-commitment verify batch: more than 2^16 openings, or more than 2^24 key elements in all");
  size_t sum = 0;
  for (size_t k = 0; k < count; k++) {
    if (proof_lens[k] > proofs_len - sum)
      return fail(RIPP_ERR_ARG, "proof_lens add up to more than proofs_len = " + std::to_string(proofs_len));
    sum += proof_lens[k];
  }
  if (sum != proofs_len)
    return fail(RIPP_ERR_ARG, "proof_lens add up to " + std::to_string(sum) + ", not proofs_len = " + std::to_string(proofs_len));
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t K = count, L2 = trusted ? 0 : log2_pow2(n), L1 = trusted ? 0 : log2_pow2(m);
  const Fq12* coms = (const Fq12*)com_gts;
  const Fr *xs = (const Fr*)x_host, *ys = (const Fr*)y_host, *evs = (const Fr*)evals;

  // ---- decoding, subgroup checks (stage A at word 2k, stage B at 2k + 1) and the host chains while they run ----
  std::vector<PcVerifyItem> it(K);
  std::vector<SubgroupSrc> src;
  for (size_t k = 0, off = 0; k < K; off += proof_lens[k], k++) {
    PcVerifyItem& a = it[k];
    pc_verify_parse(a, trusted, n, coms[k], evs[k], proofs + off, proof_lens[k]);
    if (a.status != RIPP_AGG_OK) continue;
    for (int i = 0; i < 4; i++)
      if (i < 2 || a.b_ok) src.push_back(SubgroupSrc{&a.r[i], (uint32_t)(2 * k + i / 2)});
  }
  std::vector<uint32_t> bad;
  OK(batch_subgroups(ctx, src, 2 * K, [&] {
    host_parallel(K, 4, [&](size_t k) {
      if (it[k].status == RIPP_AGG_OK && it[k].b_ok) pc_verify_host(it[k], trusted, L2, L1, xs[k], ys[k]);
    });
  }, &bad));
  // ripp_pc_verify's order: stage A's decoding, its subgroups, stage B's decoding, its subgroups, the checks
  for (size_t k = 0; k < K; k++) {
    PcVerifyItem& a = it[k];
    if (a.status == RIPP_AGG_MALFORMED) continue;
    if (bad[2 * k])
      a.status = RIPP_AGG_NOT_IN_SUBGROUP;
    else if (!a.b_ok)
      a.status = RIPP_AGG_MALFORMED;
    else if (bad[2 * k + 1])
      a.status = RIPP_AGG_NOT_IN_SUBGROUP;
  }

  // ---- every group identity of the openings still OK, in one set of launches ----
  size_t LG = 1, LD = 1;  // longest GT fold, longest G1 identity
  bool any = false;
  for (const PcVerifyItem& a : it) {
    if (a.status != RIPP_AGG_OK) continue;
    any = true;
    const size_t r2 = a.t2.size();
    LG = std::max(LG, 2 * r2 + 1);
    LD = std::max(LD, 2 * std::max(r2, a.t1.size()) + 2);
  }
  if (!any) {
    for (size_t k = 0; k < K; k++) status_out[k] = it[k].status;
    return RIPP_OK;
  }
  // equations: trusted [base (K) | final key KZG (K) | KZG at y (K)], transparent [base (K)]; the base checks' targets
  // are the GT folds.  G1 identities: trusted [K], transparent [b0 (K) | ssm (K) | first tier (K)], LD terms each.
  const size_t E = (trusted ? 3 : 1) * K, ND = (trusted ? 1 : 3) * K;
  const size_t o_D = 9 * E, nT = o_D + ND * LD;
  const size_t o_ts = up256(nT * 96), o_q = o_ts + up256(nT * 32), o_ge = o_q + up256(3 * E * 192), o_gs = o_ge + up256(K * LG * 576),
               o_tg = o_gs + up256(K * LG * 32), o_t2 = o_tg + up256(E * 576), o_t1 = o_t2 + up256(K * L2 * 32),
               o_f1 = o_t1 + up256(K * L1 * 32), hbytes = o_f1 + up256(K * 32);
  std::vector<uint8_t> H(hbytes);
  G1Aff* TB = (G1Aff*)H.data();
  Fr* TS = (Fr*)(H.data() + o_ts);
  G2Aff* Q = (G2Aff*)(H.data() + o_q);
  Fq12* GE = (Fq12*)(H.data() + o_ge);
  Fr* GS = (Fr*)(H.data() + o_gs);
  Fq12* TG = (Fq12*)(H.data() + o_tg);
  Fr *T2 = (Fr*)(H.data() + o_t2), *T1 = (Fr*)(H.data() + o_t1), *F1 = (Fr*)(H.data() + o_f1);
  const Fr one = Fr::one(), m_one = -Fr::one();
  for (size_t i = 0; i < K * LG; i++) GE[i] = Fq12::one();
  for (size_t e = K; e < E; e++) TG[e] = Fq12::one();
  auto term = [&](size_t j, size_t e, int t, const G1Aff& b, const Fr& s) {
    TB[(j * E + e) * 3 + t] = b;
    TS[(j * E + e) * 3 + t] = s;
  };
  std::vector<Val> el;
  std::vector<Fr> sc;
  // identity d: the fold's terms, then (b, s) at `at` (after the fold when at == 0)
  auto identity = [&](size_t d, const G1Aff* b, const Fr& s, size_t at) {
    for (size_t i = 0; i < el.size(); i++) {
      memcpy(&TB[o_D + d * LD + i], el[i].raw, 96);
      TS[o_D + d * LD + i] = sc[i];
    }
    const size_t i = at ? at : el.size();
    if (b) TB[o_D + d * LD + i] = *b;
    TS[o_D + d * LD + i] = s;
  };
  auto gt_fold = [&](size_t k) {
    for (size_t i = 0; i < el.size(); i++) {
      memcpy(&GE[k * LG + i], el[i].raw, 576);
      GS[k * LG + i] = sc[i];
    }
  };
  const VerifierSRS vs = trusted ? load_vsrs(vsrs) : VerifierSRS{};
  for (size_t k = 0; k < K; k++) {
    const PcVerifyItem& a = it[k];
    if (a.status != RIPP_AGG_OK) continue;
    if (trusted) {
      const GipaProofP& g = a.tp.gipa;
      const G1Aff& a0 = *(const G1Aff*)g.a0.raw;
      const G2Aff& ck = *(const G2Aff*)a.tp.ck_a.raw;
      term(0, k, 0, a0, one);
      Q[k] = ck;
      size_t e = K + k;
      term(0, e, 0, vs.g, one);
      Q[e] = ck;
      term(1, e, 0, vs.g, -a.fa);
      Q[E + e] = vs.h;
      term(2, e, 0, vs.g, a.z);
      term(2, e, 1, vs.g_beta, m_one);
      Q[2 * E + e] = a.tp.pi_a;
      e = 2 * K + k;
      term(0, e, 0, a.ye, one);
      term(0, e, 1, vs.g, -evs[k]);
      term(0, e, 2, a.pik, ys[k]);
      Q[e] = vs.h;
      term(1, e, 0, a.pik, m_one);
      Q[E + e] = vs.h_alpha;
      fold_terms(g, a.c2, a.ci2, a.com2[2], 2, &el, &sc);
      identity(k, &a0, -a.ssm2, 0);
      fold_terms(g, a.c2, a.ci2, a.com2[0], 0, &el, &sc);
      gt_fold(k);
      continue;
    }
    const G1Aff& a0 = *(const G1Aff*)a.p2.a0.raw;
    term(0, k, 0, a0, one);  // Q[k] = ck2, from the G2 MSM
    fold_terms(a.p2, a.c2, a.ci2, a.com2[2], 2, &el, &sc);
    identity(k, &a0, -*(const Fr*)a.p2.b0.raw, 0);
    identity(K + k, &a0, -a.ssm2, 0);
    fold_terms(a.p1, a.c1, a.ci1, a.com1[0], 0, &el, &sc);
    identity(2 * K + k, nullptr, m_one, LD - 1);  // the point a0 ck1 comes from the G1 MSM
    fold_terms(a.p2, a.c2, a.ci2, a.com2[0], 0, &el, &sc);
    gt_fold(k);
    for (size_t j = 0; j < L2; j++) T2[k * L2 + j] = a.t2[j].inv();
    for (size_t j = 0; j < L1; j++) T1[k * L1 + j] = a.t1[j].inv();
    F1[k] = *(const Fr*)a.p1.a0.raw;
  }

  // device: [scaled terms | P (3 x E) | G1 identities (ND) | Miller values (E) | verdicts (E) | transparent: exponents
  // of the final keys (K n, K m) | a0 ck1 (K)]
  const size_t o_P = up256(nT * 96), o_id = o_P + up256(3 * E * 96), o_ml = o_id + up256(ND * 96), o_ok = o_ml + up256(E * 576),
               o_e2 = o_ok + up256(E), o_e1 = o_e2 + (trusted ? 0 : up256(K * n * 32)), o_ck1 = o_e1 + (trusted ? 0 : up256(K * m * 32)),
               dbytes = o_ck1 + (trusted ? 0 : up256(K * 96));
  void *hd, *dd;
  OK(scratch(ctx, 39, hbytes, &hd));
  OK(scratch(ctx, 40, dbytes, &dd));
  uint8_t *Dh = (uint8_t*)hd, *Dd = (uint8_t*)dd;
  const G1Aff* scaled = (const G1Aff*)Dd;
  CU(cudaMemcpyAsync(Dh, H.data(), hbytes, cudaMemcpyHostToDevice, st));
  if (!trusted) {
    Fr *e2 = (Fr*)(Dd + o_e2), *e1 = (Fr*)(Dd + o_e1);
    k_pc_key_exponents_seg<<<(unsigned)((K * n + 127) / 128), 128, 0, st>>>((const Fr*)(Dh + o_t2), (unsigned)L2, nullptr, K, e2);
    LAUNCHED(ctx);
    OK(ripp_msm_batch_internal(ctx, 2, second_tier_dev, 0, e2, n, n, K, Dh + o_q));
    k_pc_key_exponents_seg<<<(unsigned)((K * m + 127) / 128), 128, 0, st>>>((const Fr*)(Dh + o_t1), (unsigned)L1,
                                                                          (const Fr*)(Dh + o_f1), K, e1);
    LAUNCHED(ctx);
    OK(ripp_msm_batch_internal(ctx, 1, first_tier_dev, 0, e1, m, m, K, Dd + o_ck1));
    // into the last term of every first-tier identity: one strided copy
    CU(cudaMemcpy2DAsync(Dh + (o_D + 2 * K * LD + LD - 1) * 96, LD * 96, Dd + o_ck1, 96, 96, K, cudaMemcpyDeviceToDevice, st));
  }
  OK(ripp_g1_scale_dev(ctx, Dh, Dh + o_ts, nT, Dd));
  OK(ripp_seg_sum_dev(ctx, 1, scaled, 3, (int)(3 * E), Dd + o_P));
  OK(ripp_seg_sum_dev(ctx, 1, scaled + o_D, LD, (int)ND, Dd + o_id));
  OK(ripp_gt_multiexp_l6(ctx, Dh + o_ge, Dh + o_gs, LG, Dh + o_tg, (int)K));
  OK(ripp_pairing_checks_l6(ctx, Dd + o_P, Dh + o_q, E, Dd + o_ml, Dh + o_tg, Dd + o_ok));
  std::vector<uint8_t> ok(E);
  std::vector<G1Aff> id(ND);
  CU(cudaMemcpyAsync(ok.data(), Dd + o_ok, E, cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(id.data(), Dd + o_id, ND * 96, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  size_t acc = 0;
  for (size_t k = 0; k < K; k++) {
    PcVerifyItem& a = it[k];
    if (a.status == RIPP_AGG_OK) {
      const bool pass = trusted ? ok[k] && ok[K + k] && ok[2 * K + k] && id[k].is_inf()
                                : ok[k] && id[k].is_inf() && id[K + k].is_inf() && id[2 * K + k].is_inf();
      a.status = pass ? RIPP_AGG_OK : RIPP_AGG_REJECTED;
    }
    status_out[k] = a.status;
    acc += a.status == RIPP_AGG_OK;
  }
  *n_accepted = acc;
  return RIPP_OK;
}
