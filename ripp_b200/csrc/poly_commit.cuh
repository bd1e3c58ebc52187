// The polynomial-commitment application (ip_proofs/src/applications/poly_commit/mod.rs: KZG :52-131,
// BivariatePolynomialCommitment :153-284; transparent.rs:85-213) behind the C ABI.  Part of the gipa.cu translation
// unit: the openings call its resident provers (gipa_prove, tipa_prove) and the verifiers of verify.cuh.
//
// A bivariate polynomial is one device array of `len` Fr read row-major with row length m = y_degree + 1
// (coefficient j of Y polynomial i at i m + j, zeros from `len` on), n = x_degree + 1 rows.  Its new scalar work runs
// on the device (pc_scan.cuh has the rules):
//   - the row combination y_eval[j] = sum_i x^i C[i m + j] (mod.rs:221-241), Horner over the rows with threads on
//     consecutive columns; the rows are cut into groups whose partial sums are recombined with x^R, so that a short
//     row length (the transparent skew) still fills the GPU;
//   - the division by (X - z) (mod.rs:98-104) as a chunked scan of the linear recurrence s_k = c_k + z s_(k+1): chunk
//     heads, the same scan over the heads at z^L, and a replay of every chunk from its carry.  The remainder s_0 is
//     the evaluation.
#include "pc_scan.cuh"

int ripp_fr_power_seq_internal(ripp_ctx* ctx, const Fr& s, size_t n, void* out_dev);  // setup.cu: out[i] = s^i

static const size_t PC_CHUNK = 32;      // L: coefficients per thread of the division scan
static const size_t PC_ROW_THREADS = 1 << 16;  // threads the row combination aims for (columns x row groups)

__global__ void k_pc_div_heads(const Fr* __restrict__ c, size_t N, Fr z, Fr* __restrict__ heads) {
  size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = b * PC_CHUNK;
  if (lo >= N) return;
  size_t hi = lo + PC_CHUNK < N ? lo + PC_CHUNK : N;
  heads[b] = pc::chunk_head(c, lo, hi, z, Fr::zero());
}

// S: the scan's values at the chunk starts (NULL when there is one chunk)
__global__ void k_pc_div_replay(const Fr* __restrict__ c, size_t N, Fr z, const Fr* __restrict__ S, Fr* out0, Fr* out) {
  size_t b = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = b * PC_CHUNK;
  if (lo >= N) return;
  size_t hi = lo + PC_CHUNK < N ? lo + PC_CHUNK : N;
  pc::chunk_replay(c, lo, hi, z, hi < N ? S[b + 1] : Fr::zero(), out0, out);
}

// part[g m + j] = sum_{i in [g R, (g+1) R) and i < n} x^(i - g R) C[i m + j], zero past len
__global__ void k_pc_rows(const Fr* __restrict__ C, size_t len, size_t m, size_t n, size_t R, Fr x, Fr* __restrict__ part) {
  size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  size_t g = blockIdx.y, lo = g * R, hi = lo + R < n ? lo + R : n;
  Fr acc = Fr::zero();
  for (size_t i = hi; i-- > lo;) {
    size_t at = i * m + j;
    acc = pc::horner_step(acc, x, at < len ? C[at] : Fr::zero());
  }
  part[g * m + j] = acc;
}

// y[j] = sum_g x^(g R) part[g m + j]
__global__ void k_pc_rows_combine(const Fr* __restrict__ part, size_t m, size_t G, Fr x_pow_r, Fr* __restrict__ y) {
  size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  Fr acc = Fr::zero();
  for (size_t g = G; g-- > 0;) acc = pc::horner_step(acc, x_pow_r, part[g * m + j]);
  y[j] = acc;
}

// Fr of workspace div_scan needs for N coefficients: heads and carries of every level
static size_t div_tmp_len(size_t N) {
  size_t t = 0;
  while (N > PC_CHUNK) {
    N = (N + PC_CHUNK - 1) / PC_CHUNK;
    t += 2 * N;
  }
  return t;
}

// s_k of the recurrence over c[0, N) at z (N >= 1): s_0 to out0, s_k to out[k - 1]; out must not overlap c
static int div_scan(ripp_ctx* ctx, const Fr* c, size_t N, const Fr& z, Fr* tmp, Fr* out0, Fr* out) {
  const size_t nb = (N + PC_CHUNK - 1) / PC_CHUNK;
  const unsigned blocks = (unsigned)((nb + 127) / 128);
  Fr* S = nullptr;
  if (nb > 1) {
    Fr* heads = tmp;
    S = tmp + nb;
    k_pc_div_heads<<<blocks, 128, 0, ctx->stream>>>(c, N, z, heads);
    LAUNCHED(ctx);
    OK(div_scan(ctx, heads, nb, pc::pow(z, PC_CHUNK), tmp + 2 * nb, S, S + 1));
  }
  k_pc_div_replay<<<blocks, 128, 0, ctx->stream>>>(c, N, z, S, out0, out);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// q = (f - f(z)) / (X - z) (len - 1 Fr) and f(z) (one Fr), device; tmp: div_tmp_len(len) Fr
static int div_linear(ripp_ctx* ctx, const Fr* c, size_t len, const Fr& z, Fr* tmp, Fr* q, Fr* eval) {
  if (len == 0) {
    CU(cudaMemsetAsync(eval, 0, sizeof(Fr), ctx->stream));
    return RIPP_OK;
  }
  return div_scan(ctx, c, len, z, tmp, eval, q);
}

// G groups of R rows for the row combination
static void row_groups(size_t n, size_t m, size_t* G, size_t* R) {
  size_t g = PC_ROW_THREADS / m;
  if (g < 1) g = 1;
  if (g > n) g = n;
  *R = (n + g - 1) / g;
  *G = (n + *R - 1) / *R;
}
// y[j] = sum_i x^i C[i m + j] over n rows, zeros from len on; part: G m Fr (unused when G == 1)
static int row_combination(ripp_ctx* ctx, const Fr* C, size_t len, size_t m, size_t n, const Fr& x, Fr* part, Fr* y) {
  size_t G, R;
  row_groups(n, m, &G, &R);
  dim3 grid((unsigned)((m + 127) / 128), (unsigned)G);
  k_pc_rows<<<grid, 128, 0, ctx->stream>>>(C, len, m, n, R, x, G == 1 ? y : part);
  LAUNCHED(ctx);
  if (G == 1) return RIPP_OK;
  k_pc_rows_combine<<<grid.x, 128, 0, ctx->stream>>>(part, m, G, pc::pow(x, R), y);
  LAUNCHED(ctx);
  return RIPP_OK;
}

static Fr fr_host(const void* p) {
  Fr f;
  memcpy(f.v, p, sizeof(Fr));
  return f;
}

// n rows of m: powers of two, the segmented MSM's limits, len within the rectangle
static int pc_shape(size_t n, size_t m, size_t len) {
  if (n == 0 || (n & (n - 1)) || m == 0 || (m & (m - 1)))
    return fail(RIPP_ERR_NOT_POW2, "rows, row length: " + std::to_string(n) + ", " + std::to_string(m) + " (both must be powers of two)");
  if (n > ((size_t)1 << 16) || n * m > ((size_t)1 << 24))
    return fail(RIPP_ERR_ARG, "polynomial commitment: more than 2^16 rows or 2^24 coefficients");
  if (len > n * m) return fail(RIPP_ERR_ARG, "polynomial commitment: len > rows x row length");
  return RIPP_OK;
}

extern "C" int ripp_fr_div_linear_dev(ripp_ctx* ctx, const void* coeffs_dev, size_t len, const void* z_host, void* q_out_dev,
                                      void* eval_out_dev) {
  if (!ctx || !z_host || (len && !coeffs_dev) || (len > 1 && !q_out_dev)) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  const size_t nt = div_tmp_len(len);
  void* d;
  OK(scratch(ctx, 45, (nt + 1) * sizeof(Fr), &d));
  Fr* ev = eval_out_dev ? (Fr*)eval_out_dev : (Fr*)d + nt;
  return div_linear(ctx, (const Fr*)coeffs_dev, len, fr_host(z_host), (Fr*)d, (Fr*)q_out_dev, ev);
}

// ------------------------------------------------------------------------------------------------
// KZG (mod.rs:52-131)
// ------------------------------------------------------------------------------------------------
extern "C" int ripp_pc_kzg_commit_dev(ripp_ctx* ctx, const void* powers_dev, size_t n_powers, const void* coeffs_dev, size_t len,
                                      void* g1_aff_out_dev) {
  if (!ctx || !g1_aff_out_dev || (len && (!powers_dev || !coeffs_dev))) return fail(RIPP_ERR_ARG, "null argument");
  if (len > n_powers) return fail(RIPP_ERR_ARG, "KZG: more coefficients than powers (mod.rs:85)");
  return ripp_msm_g1_dev(ctx, powers_dev, coeffs_dev, len, g1_aff_out_dev);
}

extern "C" int ripp_pc_kzg_open_dev(ripp_ctx* ctx, const void* powers_dev, size_t n_powers, const void* coeffs_dev, size_t len,
                                    const void* z_host, void* g1_aff_out_dev, void* eval_out_dev) {
  if (!ctx || !z_host || !g1_aff_out_dev || (len && (!powers_dev || !coeffs_dev))) return fail(RIPP_ERR_ARG, "null argument");
  if (len > n_powers) return fail(RIPP_ERR_ARG, "KZG: more coefficients than powers (mod.rs:98)");
  CU(cudaSetDevice(ctx->device));
  const size_t nt = div_tmp_len(len), nq = len ? len - 1 : 0;
  void* d;
  OK(scratch(ctx, 45, (nt + nq + 1) * sizeof(Fr), &d));
  Fr* q = (Fr*)d + nt;
  Fr* ev = eval_out_dev ? (Fr*)eval_out_dev : q + nq;
  OK(div_linear(ctx, (const Fr*)coeffs_dev, len, fr_host(z_host), (Fr*)d, q, ev));
  return ripp_msm_g1_dev(ctx, powers_dev, q, nq, g1_aff_out_dev);  // no quotient (len <= 1): the identity
}

// mod.rs:120-130: e(com - g eval, h) == e(proof, h_alpha - h z), as e(com - g eval, h) e(-proof, h_alpha - h z) == 1
static int kzg_verify(ripp_ctx* ctx, const VerifierSRS& vs, const G1Aff& com, const Fr& z, const Fr& eval, const G1Aff& proof,
                      bool* okp) {
  void* d;
  OK(scratch(ctx, 45, 4096, &d));
  char* D = (char*)d;
  char *g1 = D, *g2 = D + 1024, *res = D + 2048;
  cudaStream_t st = ctx->stream;
  G1Aff neg = proof.is_inf() ? proof : proof.neg();
  CU(cudaMemcpyAsync(g1, &vs.g, 96, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(g1 + 96, &com, 96, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(g1 + 192, &neg, 96, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(g2, &vs.h, 192, cudaMemcpyHostToDevice, st));
  CU(cudaMemcpyAsync(g2 + 192, &vs.h_alpha, 192, cudaMemcpyHostToDevice, st));
  Fr m_eval = -eval, m_z = -z;
  OK(ripp_g1_fold_dev(ctx, g1, g1 + 96, m_eval.v, 1, g1 + 96));   // com - g eval
  OK(ripp_g2_fold_dev(ctx, g2, g2 + 192, m_z.v, 1, g2 + 192));    // h_alpha - h z
  OK(ripp_pairing_ip_dev(ctx, g1 + 96, g2, 2, res));
  Fq12 out;
  CU(cudaMemcpyAsync(&out, res, 576, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  Fq12 one = Fq12::one();
  *okp = memcmp(&out, &one, 576) == 0;
  return RIPP_OK;
}

extern "C" int ripp_pc_kzg_verify(ripp_ctx* ctx, const void* vsrs, const void* com, const void* z, const void* eval,
                                  const void* proof, int* accept) {
  if (!ctx || !vsrs || !com || !z || !eval || !proof || !accept) return fail(RIPP_ERR_ARG, "null argument");
  *accept = 0;
  CU(cudaSetDevice(ctx->device));
  G1Aff c, p;
  memcpy(&c, com, 96);
  memcpy(&p, proof, 96);
  bool ok = false;
  OK(kzg_verify(ctx, load_vsrs(vsrs), c, fr_host(z), fr_host(eval), p, &ok));
  *accept = ok ? 1 : 0;
  return RIPP_OK;
}

// ------------------------------------------------------------------------------------------------
// bivariate commitments, trusted (mod.rs:153-284) and transparent (transparent.rs:85-213)
// ------------------------------------------------------------------------------------------------
// mod.rs:186 / transparent.rs:106-119: the n Y polynomials' first-tier commitments (KZG over the powers, or
// Pedersen over the first-tier key: both one MSM over m shared bases) as ONE segmented MSM, then the AFGHO pairing
// product with the second-tier key.
extern "C" int ripp_pc_commit_dev(ripp_ctx* ctx, const void* first_tier_dev, size_t m, const void* second_tier_dev, size_t n,
                                  const void* coeffs_dev, size_t len, void* gt_out, void* y_coms_dev) {
  if (!ctx || !first_tier_dev || !second_tier_dev || !gt_out || !y_coms_dev || (len && !coeffs_dev))
    return fail(RIPP_ERR_ARG, "null argument");
  OK(pc_shape(n, m, len));
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const void* sc = coeffs_dev;
  void* d;
  OK(scratch(ctx, 47, (len < n * m ? n * m * sizeof(Fr) : 0) + 1024, &d));
  char* res = (char*)d;
  if (len < n * m) {  // the rows past len are zero: one padded copy, whatever the number of rows
    char* pad = (char*)d + 1024;
    if (len) CU(cudaMemcpyAsync(pad, coeffs_dev, len * sizeof(Fr), cudaMemcpyDeviceToDevice, st));
    CU(cudaMemsetAsync(pad + len * sizeof(Fr), 0, (n * m - len) * sizeof(Fr), st));
    sc = pad;
  }
  OK(ripp_msm_batch_internal(ctx, 1, first_tier_dev, 0, sc, m, m, n, y_coms_dev));
  OK(ripp_pairing_ip_dev(ctx, y_coms_dev, second_tier_dev, n, res));
  CU(cudaMemcpyAsync(gt_out, res, 576, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return RIPP_OK;
}

extern "C" int ripp_pc_open_dev(ripp_ctx* ctx, int kind, const void* first_tier_dev, size_t m, const void* second_tier_dev,
                                size_t n, const void* srs_g2_dev, const void* coeffs_dev, size_t len, const void* y_coms_dev,
                                const void* x_host, const void* y_host, uint8_t* proof_out, size_t proof_cap, size_t* proof_len,
                                void* eval_out) {
  if (!ctx || !first_tier_dev || !second_tier_dev || !y_coms_dev || !x_host || !y_host || (len && !coeffs_dev))
    return fail(RIPP_ERR_ARG, "null argument");
  if (kind != RIPP_PC_TRUSTED && kind != RIPP_PC_TRANSPARENT) return fail(RIPP_ERR_ARG, "bad polynomial-commitment kind");
  if (kind == RIPP_PC_TRUSTED && !srs_g2_dev) return fail(RIPP_ERR_ARG, "the trusted opening needs h_beta_powers");
  OK(pc_shape(n, m, len));
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const Fr x = fr_host(x_host), y = fr_host(y_host);
  size_t G, R;
  row_groups(n, m, &G, &R);
  // workspace: powers of x (n) | y_eval (m) | powers of y or the quotient (m) | row partials (G m) | scan (div) |
  // eval (1) | y_eval_comm, kzg proof (2 G1)
  const size_t o_px = 0, o_ye = o_px + n, o_q = o_ye + m, o_part = o_q + m, o_tmp = o_part + (G > 1 ? G * m : 0),
               o_ev = o_tmp + div_tmp_len(m), o_end = o_ev + 1;
  void* d;
  OK(scratch(ctx, 44, o_end * sizeof(Fr) + 2 * sizeof(G1Aff), &d));
  Fr* F = (Fr*)d;
  G1Aff* pts = (G1Aff*)(F + o_end);
  // mod.rs:221-241 and the transparent open after :137: powers of x, y_eval, y_eval_comm
  OK(ripp_fr_power_seq_internal(ctx, x, n, F + o_px));
  OK(row_combination(ctx, (const Fr*)coeffs_dev, len, m, n, x, F + o_part, F + o_ye));
  OK(ripp_msm_g1_dev(ctx, first_tier_dev, F + o_ye, m, pts));
  if (kind == RIPP_PC_TRUSTED) {
    // kzg_proof = KZG::open(kzg, y_eval, y) (mod.rs:98-104): quotient (m - 1 coefficients) and y_eval(y) = f(x, y)
    OK(div_linear(ctx, F + o_ye, m, y, F + o_tmp, F + o_q, F + o_ev));
    OK(ripp_msm_g1_dev(ctx, first_tier_dev, F + o_q, m - 1, pts + 1));
  } else {
    // transparent first tier: powers of y, and f(x, y) = <y_eval, powers of y>
    OK(ripp_fr_power_seq_internal(ctx, y, m, F + o_q));
    OK(ripp_scalar_ip_dev(ctx, F + o_ye, F + o_q, m, F + o_ev));
  }
  G1Aff host_pts[2];
  Fr ev;
  CU(cudaMemcpyAsync(host_pts, pts, sizeof(host_pts), cudaMemcpyDeviceToHost, st));
  CU(cudaMemcpyAsync(&ev, F + o_ev, sizeof(Fr), cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  Bytes proof;
  if (kind == RIPP_PC_TRUSTED) {
    // TIPAWithSSM over (y_coms, powers of x) with the second-tier key; OpeningProof (mod.rs:145-149):
    // ip_proof || y_eval_comm || kzg_proof
    OK(tipa_prove(ctx, RIPP_GIPA_MULTIEXP_SSM, nullptr, srs_g2_dev, y_coms_dev, F + o_px, second_tier_dev, nullptr, n, Fr::one(),
                  &proof));
    put_g1(proof, host_pts[0]);
    put_g1(proof, host_pts[1]);
  } else {
    // second-tier GIPA (MULTIEXP_SSM), first-tier GIPA (SCALAR_SSM_G1 on y_eval, powers of y);
    // OpeningProof (:79-83): second_tier_ip_proof || y_eval_comm || first_tier_ip_proof
    GipaSpec s2, s1;
    gipa_spec(RIPP_GIPA_MULTIEXP_SSM, &s2);
    gipa_spec(RIPP_GIPA_SCALAR_SSM_G1, &s1);
    GipaOut g2, g1;
    OK(gipa_prove(ctx, s2, y_coms_dev, F + o_px, second_tier_dev, nullptr, n, &g2));
    OK(gipa_prove(ctx, s1, F + o_ye, F + o_q, first_tier_dev, nullptr, m, &g1));
    proof = g2.proof;
    put_g1(proof, host_pts[0]);
    proof.insert(proof.end(), g1.proof.begin(), g1.proof.end());
  }
  if (eval_out) memcpy(eval_out, &ev, sizeof(Fr));
  return copy_out(proof, proof_out, proof_cap, proof_len);
}

// GIPAProof length of the transparent second tier for n = 2^k keys (MULTIEXP_SSM as gipa_prove writes it): u64 round
// count, per round com_1 and com_2 = (GT, Fr placeholder, IdentityOutput<G1>), then r_base = (G1, Fr)
static size_t transparent_second_len(size_t n) {
  size_t k = 0;
  while (((size_t)1 << k) < n) k++;
  return 8 + k * 2 * (576 + 32 + 8 + 96) + 96 + 32;
}

extern "C" int ripp_pc_verify(ripp_ctx* ctx, int kind, const void* vsrs, const void* first_tier_dev, size_t m,
                              const void* second_tier_dev, size_t n, const void* com_gt, const void* x_host, const void* y_host,
                              const void* eval, const uint8_t* proof, size_t proof_len, int* accept) {
  if (!ctx || !accept || !com_gt || !x_host || !y_host || !eval || !proof) return fail(RIPP_ERR_ARG, "null argument");
  *accept = 0;
  if (kind != RIPP_PC_TRUSTED && kind != RIPP_PC_TRANSPARENT) return fail(RIPP_ERR_ARG, "bad polynomial-commitment kind");
  CU(cudaSetDevice(ctx->device));
  const Fr ev = fr_host(eval);
  if (kind == RIPP_PC_TRUSTED) {
    // BivariatePolynomialCommitment::verify: TIPAWithSSM on com || IdentityOutput(y_eval_comm) at x, then KZG::verify(y_eval_comm) at y
    if (!vsrs) return fail(RIPP_ERR_ARG, "null argument");
    if (proof_len < 192) return fail(RIPP_ERR_ARG, "malformed OpeningProof bytes");
    const uint8_t* ye = proof + proof_len - 192;
    Reader rp(ye, 192);
    G1Aff y_eval_comm, kzg_proof;
    if (!get_g1(rp, &y_eval_comm) || !get_g1(rp, &kzg_proof) || !rp.done()) return fail(RIPP_ERR_ARG, "malformed OpeningProof bytes");
    uint32_t bad = 0;
    OK(validate_subgroups(ctx, {&rp}, &bad));
    if (bad) return subgroup_error(bad);
    Bytes com;
    put_gt(com, *(const Fq12*)com_gt);
    put_u64_le(com, 1);
    com.insert(com.end(), ye, ye + 96);
    int ip_ok = 0;
    OK(ripp_tipa_verify(ctx, RIPP_GIPA_MULTIEXP_SSM, vsrs, com.data(), com.size(), x_host, proof, proof_len - 192, &ip_ok));
    bool kzg_ok = false;
    OK(kzg_verify(ctx, load_vsrs(vsrs), y_eval_comm, fr_host(y_host), ev, kzg_proof, &kzg_ok));
    *accept = ip_ok && kzg_ok ? 1 : 0;
    return RIPP_OK;
  }
  // TransparentBivariatePolynomialCommitment::verify: the two GIPAs with structured scalar message
  if (!first_tier_dev || !second_tier_dev) return fail(RIPP_ERR_ARG, "null argument");
  OK(pc_shape(n, m, 0));
  const size_t s = transparent_second_len(n);
  if (proof_len < s + 96) return fail(RIPP_ERR_ARG, "malformed OpeningProof bytes");
  const uint8_t* ye = proof + s;
  Bytes st2, st1;
  put_gt(st2, *(const Fq12*)com_gt);
  put_u64_le(st2, 1);
  st2.insert(st2.end(), ye, ye + 96);
  st1.insert(st1.end(), ye, ye + 96);
  put_u64_le(st1, 1);
  put_fr(st1, ev);
  int ok2 = 0, ok1 = 0;
  OK(ripp_gipa_verify_dev(ctx, RIPP_GIPA_MULTIEXP_SSM, second_tier_dev, nullptr, n, st2.data(), st2.size(), x_host, proof, s, &ok2));
  OK(ripp_gipa_verify_dev(ctx, RIPP_GIPA_SCALAR_SSM_G1, first_tier_dev, nullptr, m, st1.data(), st1.size(), y_host, ye + 96,
                          proof_len - s - 96, &ok1));
  *accept = ok2 && ok1 ? 1 : 0;
  return RIPP_OK;
}
