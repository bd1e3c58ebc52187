// Groth16 verification with one verdict per proof (include/ripp_b200.h "Groth16 verification"): ark-groth16 0.4
// prepare_verifying_key, prepare_inputs and verify_proof for batches of proofs, from device limbs or from untrusted
// ark-serialize bytes.  The kernels live with their engines: the fixed-base tables and prepare_inputs in setup.cu, the
// per-proof Miller loops and the final exponentiation with its compare in pairing6.cu.
#include "common.cuh"
#include "rlc.cuh"
#include "serde.cuh"

// Prepared key (device): e(alpha, beta) | -gamma | -delta | IC_0 | the fixed-base tables of IC_1..IC_m
constexpr size_t PVK_NG = 576, PVK_ND = PVK_NG + 192, PVK_IC0 = PVK_ND + 192, PVK_TAB = 1280;
// packed host verifying key (ripp_tipp_verify_aggregate): alpha_g1 | beta_g2 | gamma_g2 | delta_g2 | gamma_abc_g1[m + 1]
constexpr size_t VK_BETA = 96, VK_GAMMA = VK_BETA + 192, VK_DELTA = VK_GAMMA + 192, VK_IC = VK_DELTA + 192;

__global__ void k_groth16_vk_neg(const uint8_t* __restrict__ vk, uint8_t* __restrict__ pvk) {
  if (threadIdx.x != 0) return;
  *(G2Aff*)(pvk + PVK_NG) = ((const G2Aff*)(vk + VK_GAMMA))->neg();
  *(G2Aff*)(pvk + PVK_ND) = ((const G2Aff*)(vk + VK_DELTA))->neg();
  *(G1Aff*)(pvk + PVK_IC0) = *(const G1Aff*)(vk + VK_IC);
}

// The public inputs of one proof per thread (n x m ark-serialize Fr, 32 bytes each): canonical check and Montgomery
// form; status[i] = the first failure of A, B, C (decode statuses abc[0, n), [n, 2n), [2n, 3n)), then of the inputs.
__global__ void __launch_bounds__(64) k_fr_deserialize(const uint8_t* __restrict__ in, uint32_t n, uint32_t m,
                                                       const uint8_t* __restrict__ abc, Fr* __restrict__ x,
                                                       uint8_t* __restrict__ status) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  uint8_t s = abc[i] ? abc[i] : (abc[n + i] ? abc[n + i] : abc[2 * n + i]);
  for (uint32_t j = 0; j < m; j++) {
    const size_t e = (size_t)i * m + j;
    if (!serde::decode_fr(in + 32 * e, x + e) && !s) s = RIPP_GROTH16_INPUT_NONCANONICAL;
  }
  status[i] = s;
}

extern "C" size_t ripp_groth16_pvk_bytes(size_t m) { return PVK_TAB + m * ripp_groth16_table_bytes(); }

extern "C" int ripp_groth16_prepare_vk_dev(ripp_ctx* ctx, const void* vk, size_t m, void* pvk_dev) {
  if (!ctx || !vk || !pvk_dev) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  const size_t vk_bytes = VK_IC + (m + 1) * 96;
  void* d;
  OK(scratch(ctx, 32, vk_bytes, &d));
  uint8_t *V = (uint8_t*)d, *K = (uint8_t*)pvk_dev;
  CU(cudaMemcpyAsync(V, vk, vk_bytes, cudaMemcpyHostToDevice, ctx->stream));
  OK(ripp_pairing_ip_dev(ctx, V, V + VK_BETA, 1, K));  // e(alpha, beta): the eighteen-lane path at n = 1
  k_groth16_vk_neg<<<1, 32, 0, ctx->stream>>>(V, K);
  LAUNCHED(ctx);
  OK(ripp_groth16_tables(ctx, V + VK_IC + 96, m, K + PVK_TAB));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

// P_i, the three Miller loops of each proof, the final exponentiation and the compare; `pre` as k_groth16_check6
static int verify_batch(ripp_ctx* ctx, const void* pvk, size_t m, const void* x, const void* a, const void* b, const void* c,
                        size_t n, const uint8_t* pre, uint8_t* out) {
  const size_t o_m = (n * sizeof(G1Aff) + 255) & ~(size_t)255;
  void* d;
  OK(scratch(ctx, 33, o_m + n * sizeof(Fq12), &d));
  const uint8_t* K = (const uint8_t*)pvk;
  OK(ripp_groth16_inputs(ctx, K + PVK_IC0, K + PVK_TAB, m, x, n, d));
  return ripp_groth16_pairings_l6(ctx, a, b, d, c, K + PVK_NG, K + PVK_ND, K, n, (char*)d + o_m, pre, out);
}

// argument checks of the _dev entries
static int check_dev_args(ripp_ctx* ctx, const void* pvk, size_t m, const void* x, const void* a, const void* b, const void* c,
                          size_t n, const uint8_t* out) {
  if (!ctx || !pvk || (n && (!a || !b || !c || !out || (m && !x)))) return fail(RIPP_ERR_ARG, "null argument");
  if (n > (size_t)0xffffffffu) return fail(RIPP_ERR_ARG, "more than 2^32 - 1 proofs");
  return RIPP_OK;
}

extern "C" int ripp_groth16_verify_batch_dev(ripp_ctx* ctx, const void* pvk_dev, size_t m, const void* inputs_dev,
                                             const void* a_dev, const void* b_dev, const void* c_dev, size_t n,
                                             uint8_t* verdict_dev) {
  OK(check_dev_args(ctx, pvk_dev, m, inputs_dev, a_dev, b_dev, c_dev, n, verdict_dev));
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  return verify_batch(ctx, pvk_dev, m, inputs_dev, a_dev, b_dev, c_dev, n, nullptr, verdict_dev);
}

// ---- verification by random linear combination (include/ripp_b200.h "ripp_groth16_verify_rlc_dev") -----------------
// Segments of s consecutive proofs; each segment is checked as one virtual proof,
//   final_exp( prod_i ML(r_i A_i, B_i) * ML(P_s, -gamma) * ML(C_s, -delta) ) == e(alpha, beta),
// P_s = IC_0 + sum_j sigma_sj IC_j with sigma_sj = sum_i r_i x_ij, C_s = sum_i r_i C_i, sum_i r_i = 1 (rlc.cuh).  The
// members of failing segments go through verify_batch.  A proof is a member unless the serialized entry gave it a
// decode or input status; non-members get r_i = 0.
struct RlcSeed {
  uint8_t b[32];
};

// proofs per segment: RIPP_B200_G16_RLC_SEG, default 58 -- with the two fixed-Q pairs a segment is 60 pairs, whole
// warps for every pairs-per-group count of the six-lane engine (5 KP, KP = 1..4)
static size_t rlc_seg() {
  static const long v = [] {
    const char* e = getenv("RIPP_B200_G16_RLC_SEG");
    const long s = e ? atol(e) : 0;
    return s >= 1 ? s : 58L;
  }();
  return (size_t)v;
}

// one thread per ChaCha20 block (four proofs); r[i] = 0 for non-members (pre[i] != 0)
__global__ void __launch_bounds__(64) k_rlc_scalars(RlcSeed seed, uint32_t n, const uint8_t* __restrict__ pre,
                                                    Fr* __restrict__ r) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if ((size_t)t * 4 >= n) return;
  Fr v[4];
  rlc::scalars4(seed.b, t, v);
  for (int q = 0; q < 4; q++) {
    const uint32_t i = 4 * t + q;
    if (i < n) r[i] = pre && pre[i] ? Fr::zero() : v[q];
  }
}

static __device__ __forceinline__ Fr warp_sum(Fr a) {
  for (int o = 16; o >= 1; o >>= 1) {
    Fr b;
#pragma unroll
    for (int w = 0; w < 8; w++) b.v[w] = __shfl_xor_sync(0xffffffffu, a.v[w], o);
    a = a + b;
  }
  return a;
}

// one warp per segment: r of the last member <- 1 - sum of the others', sigma[seg][j] = sum_i r_i x_ij (j < m)
__global__ void __launch_bounds__(128) k_rlc_segment_fr(Fr* __restrict__ r, const Fr* __restrict__ x, const uint8_t* __restrict__ pre,
                                                        uint32_t n, uint32_t m, uint32_t s, uint32_t nseg, Fr* __restrict__ sigma) {
  const uint32_t seg = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (seg >= nseg) return;
  const uint32_t lo = seg * s, hi = (uint32_t)min((uint64_t)n, (uint64_t)lo + s);
  int64_t last = -1;
  for (uint32_t i = lo + lane; i < hi; i += 32)
    if (!pre || !pre[i]) last = i;
  for (int o = 16; o >= 1; o >>= 1) last = max(last, (int64_t)__shfl_xor_sync(0xffffffffu, (long long)last, o));
  if (last < 0) return;  // no member: P_s = IC_0, C_s = O, and nothing to re-check
  Fr acc = Fr::zero();
  for (uint32_t i = lo + lane; i < hi; i += 32)
    if (i != (uint32_t)last) acc = acc + r[i];  // non-members hold zero
  const Fr rl = rlc::last(warp_sum(acc));
  if (lane == 0) r[last] = rl;
  for (uint32_t j = 0; j < m; j++) {
    acc = Fr::zero();
    for (uint32_t i = lo + lane; i < hi; i += 32)
      if (!pre || !pre[i]) acc = acc + (i == (uint32_t)last ? rl : r[i]) * x[(size_t)i * m + j];
    acc = warp_sum(acc);
    if (lane == 0) sigma[(size_t)seg * m + j] = acc;
  }
}

// per proof: a member of a passing segment is accepted (out = 1, or RIPP_GROTH16_OK with `pre`, which out aliases);
// a member of a failing segment is appended to the re-check list with its A, B, C and inputs.  The list's order
// does not matter: idx carries each entry's proof index.
__global__ void __launch_bounds__(64) k_rlc_gather(const uint8_t* __restrict__ seg_ok, uint32_t n, uint32_t m, uint32_t s,
                                                   const G1Aff* __restrict__ a, const G2Aff* __restrict__ b,
                                                   const G1Aff* __restrict__ c, const Fr* __restrict__ x, const uint8_t* pre,
                                                   uint8_t* out, uint32_t* __restrict__ cnt, uint32_t* __restrict__ idx,
                                                   G1Aff* __restrict__ ga, G2Aff* __restrict__ gb, G1Aff* __restrict__ gc,
                                                   Fr* __restrict__ gx) {
  const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n || (pre && pre[i])) return;
  if (seg_ok[i / s]) {
    out[i] = pre ? (uint8_t)RIPP_GROTH16_OK : 1;
    return;
  }
  const uint32_t k = atomicAdd(cnt, 1u);
  idx[k] = i;
  ga[k] = a[i];
  gb[k] = b[i];
  gc[k] = c[i];
  for (uint32_t j = 0; j < m; j++) gx[(size_t)k * m + j] = x[(size_t)i * m + j];
}

__global__ void __launch_bounds__(64) k_rlc_scatter(const uint32_t* __restrict__ idx, const uint8_t* __restrict__ v, uint32_t k,
                                                    bool status, uint8_t* __restrict__ out) {
  const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t < k) out[idx[t]] = status ? (v[t] ? (uint8_t)RIPP_GROTH16_OK : (uint8_t)RIPP_GROTH16_REJECTED) : v[t];
}

// `pre` (serialized entry): statuses so far, members are the zeros; out receives verdicts, or statuses when pre is set
// (out may alias pre).  Synchronous: the re-check count is copied to the host before the fallback is queued.
static int verify_rlc(ripp_ctx* ctx, const void* pvk, size_t m, const void* x, const void* a, const void* b, const void* c,
                      size_t n, const uint8_t* seed32, const uint8_t* pre, uint8_t* out, size_t* n_rechecked) {
  const size_t s = rlc_seg() < n ? rlc_seg() : n, S = (n + s - 1) / s;
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t o_sig = up(n * sizeof(Fr)), o_ra = o_sig + up(S * m * sizeof(Fr) + 32), o_rc = o_ra + up(n * sizeof(G1Aff)),
               o_ps = o_rc + up(S * s * sizeof(G1Aff)), o_cs = o_ps + up(S * sizeof(G1Aff)), o_ok = o_cs + up(S * sizeof(G1Aff)),
               o_cnt = o_ok + up(S), total = o_cnt + 256;
  void* d;
  OK(scratch(ctx, 34, total, &d));
  uint8_t* D = (uint8_t*)d;
  Fr *r = (Fr*)D, *sig = (Fr*)(D + o_sig);
  G1Aff *ra = (G1Aff*)(D + o_ra), *rc = (G1Aff*)(D + o_rc), *ps = (G1Aff*)(D + o_ps), *cs = (G1Aff*)(D + o_cs);
  uint8_t* ok = D + o_ok;
  uint32_t* cnt = (uint32_t*)(D + o_cnt);
  const uint8_t* K = (const uint8_t*)pvk;
  RlcSeed sd;
  memcpy(sd.b, seed32, 32);
  {
    TimeScope ts_(ctx, RIPP_T_OTHER);
    k_rlc_scalars<<<(unsigned)((n + 255) / 256), 64, 0, ctx->stream>>>(sd, (uint32_t)n, pre, r);
    LAUNCHED(ctx);
    // sigma of a segment without members stays zero (P_s = IC_0)
    if (m) CU(cudaMemsetAsync(sig, 0, S * m * sizeof(Fr), ctx->stream));
    k_rlc_segment_fr<<<(unsigned)((S + 3) / 4), 128, 0, ctx->stream>>>(r, (const Fr*)x, pre, (uint32_t)n, (uint32_t)m, (uint32_t)s,
                                                                     (uint32_t)S, sig);
    LAUNCHED(ctx);
  }
  OK(ripp_g1_scale_dev(ctx, a, r, n, ra));
  OK(ripp_g1_scale_dev(ctx, c, r, n, rc));
  if (S * s > n) CU(cudaMemsetAsync(rc + n, 0, (S * s - n) * sizeof(G1Aff), ctx->stream));  // the identity
  {
    TimeScope ts_(ctx, RIPP_T_SCALE);
    OK(ripp_seg_sum_dev(ctx, 1, rc, s, (int)S, cs));
  }
  OK(ripp_groth16_inputs(ctx, K + PVK_IC0, K + PVK_TAB, m, sig, S, ps));
  OK(ripp_groth16_rlc_pairings_l6(ctx, ra, b, ps, cs, K + PVK_NG, K + PVK_ND, K, n, s, S, ok));
  // the fallback: members of failing segments through the per-proof path
  const size_t o_gb = up(n * sizeof(G1Aff)), o_gc = o_gb + up(n * sizeof(G2Aff)), o_gx = o_gc + up(n * sizeof(G1Aff)),
               o_idx = o_gx + up(n * m * sizeof(Fr)), o_gv = o_idx + up(n * 4), gtotal = o_gv + up(n);
  void* g;
  OK(scratch(ctx, 35, gtotal, &g));
  uint8_t* G = (uint8_t*)g;
  uint8_t* pin;
  OK(pinned(ctx, &pin));
  {
    TimeScope ts_(ctx, RIPP_T_OTHER);
    CU(cudaMemsetAsync(cnt, 0, 4, ctx->stream));
    k_rlc_gather<<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>(ok, (uint32_t)n, (uint32_t)m, (uint32_t)s, (const G1Aff*)a,
                                                                    (const G2Aff*)b, (const G1Aff*)c, (const Fr*)x, pre, out, cnt,
                                                                    (uint32_t*)(G + o_idx), (G1Aff*)G, (G2Aff*)(G + o_gb),
                                                                    (G1Aff*)(G + o_gc), (Fr*)(G + o_gx));
    LAUNCHED(ctx);
    CU(cudaMemcpyAsync(pin, cnt, 4, cudaMemcpyDeviceToHost, ctx->stream));
  }
  CU(cudaStreamSynchronize(ctx->stream));
  uint32_t k;
  memcpy(&k, pin, 4);
  *n_rechecked = k;
  if (k == 0) return RIPP_OK;
  OK(verify_batch(ctx, pvk, m, G + o_gx, G, G + o_gb, G + o_gc, k, nullptr, G + o_gv));
  TimeScope ts_(ctx, RIPP_T_OTHER);
  k_rlc_scatter<<<(k + 63) / 64, 64, 0, ctx->stream>>>((const uint32_t*)(G + o_idx), G + o_gv, k, pre != nullptr, out);
  LAUNCHED(ctx);
  return RIPP_OK;
}

extern "C" int ripp_groth16_verify_rlc_dev(ripp_ctx* ctx, const void* pvk_dev, size_t m, const void* inputs_dev, const void* a_dev,
                                           const void* b_dev, const void* c_dev, size_t n, const uint8_t* seed32,
                                           uint8_t* verdict_dev, size_t* n_rechecked) {
  if (!seed32 || !n_rechecked) return fail(RIPP_ERR_ARG, "null argument");
  OK(check_dev_args(ctx, pvk_dev, m, inputs_dev, a_dev, b_dev, c_dev, n, verdict_dev));
  *n_rechecked = 0;
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  OK(verify_rlc(ctx, pvk_dev, m, inputs_dev, a_dev, b_dev, c_dev, n, seed32, nullptr, verdict_dev, n_rechecked));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

// The serialized entries: one H2D copy of the records and one of the inputs, the decode of A, B, C and of the inputs,
// then verify_rlc with seed32 (n_rechecked set), or verify_batch without; the statuses go back to status_host.
static int verify_serialized(ripp_ctx* ctx, const void* pvk_dev, size_t m, const uint8_t* inputs_host, size_t inputs_len,
                             const uint8_t* proofs_host, size_t proofs_len, size_t n, int compressed, const uint8_t* seed32,
                             uint8_t* status_host, size_t* n_valid, size_t* n_rechecked) {
  if (!ctx || !pvk_dev || !n_valid || (n && (!proofs_host || !status_host || (m && !inputs_host))))
    return fail(RIPP_ERR_ARG, "null argument");
  if (n > (size_t)0xffffffffu) return fail(RIPP_ERR_ARG, "more than 2^32 - 1 proofs");
  const size_t rec = compressed ? 192 : 384;
  if (proofs_len != n * rec)
    return fail(RIPP_ERR_ARG, "proof bytes: " + std::to_string(proofs_len) + " bytes is not " + std::to_string(n) + " records of " +
                                  std::to_string(rec) + " bytes");
  if (m > (((size_t)1 << 40) / 32) || inputs_len != n * m * 32)
    return fail(RIPP_ERR_ARG, "input bytes: " + std::to_string(inputs_len) + " bytes is not " + std::to_string(n) + " x " +
                                  std::to_string(m) + " elements of 32 bytes");
  *n_valid = 0;
  if (seed32) *n_rechecked = 0;
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  auto up = [](size_t v) { return (v + 255) & ~(size_t)255; };
  const size_t xb = n * m * 32;
  DecodedProofs dp;
  OK(ripp_decode_proofs(ctx, proofs_host, n, compressed, 2 * up(xb) + n, &dp));
  uint8_t* xin = (uint8_t*)dp.extra;
  Fr* x = (Fr*)(xin + up(xb));
  uint8_t* st = xin + 2 * up(xb);
  if (xb) CU(cudaMemcpyAsync(xin, inputs_host, xb, cudaMemcpyHostToDevice, ctx->stream));
  k_fr_deserialize<<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>(xin, (uint32_t)n, (uint32_t)m, dp.status, x, st);
  LAUNCHED(ctx);
  if (seed32)
    OK(verify_rlc(ctx, pvk_dev, m, x, dp.a, dp.b, dp.c, n, seed32, st, st, n_rechecked));
  else
    OK(verify_batch(ctx, pvk_dev, m, x, dp.a, dp.b, dp.c, n, st, st));
  CU(cudaMemcpyAsync(status_host, st, n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  size_t ok = 0;
  for (size_t i = 0; i < n; i++) ok += status_host[i] == RIPP_GROTH16_OK;
  *n_valid = ok;
  return RIPP_OK;
}

extern "C" int ripp_groth16_verify_serialized(ripp_ctx* ctx, const void* pvk_dev, size_t m, const uint8_t* inputs_host,
                                              size_t inputs_len, const uint8_t* proofs_host, size_t proofs_len, size_t n,
                                              int compressed, uint8_t* status_host, size_t* n_valid) {
  return verify_serialized(ctx, pvk_dev, m, inputs_host, inputs_len, proofs_host, proofs_len, n, compressed, nullptr, status_host,
                           n_valid, nullptr);
}

extern "C" int ripp_groth16_verify_rlc_serialized(ripp_ctx* ctx, const void* pvk_dev, size_t m, const uint8_t* inputs_host,
                                                  size_t inputs_len, const uint8_t* proofs_host, size_t proofs_len, size_t n,
                                                  int compressed, const uint8_t* seed32, uint8_t* status_host, size_t* n_valid,
                                                  size_t* n_rechecked) {
  if (!seed32 || !n_rechecked) return fail(RIPP_ERR_ARG, "null argument");
  return verify_serialized(ctx, pvk_dev, m, inputs_host, inputs_len, proofs_host, proofs_len, n, compressed, seed32, status_host,
                           n_valid, n_rechecked);
}
