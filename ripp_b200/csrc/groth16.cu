// Groth16 verification with one verdict per proof (include/ripp_b200.h "Groth16 verification"): ark-groth16 0.4
// prepare_verifying_key, prepare_inputs and verify_proof for batches of proofs, from device limbs or from untrusted
// ark-serialize bytes.  The kernels live with their engines: the fixed-base tables and prepare_inputs in setup.cu, the
// per-proof Miller loops and the final exponentiation with its compare in pairing6.cu.
#include "common.cuh"
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

extern "C" int ripp_groth16_verify_batch_dev(ripp_ctx* ctx, const void* pvk_dev, size_t m, const void* inputs_dev,
                                             const void* a_dev, const void* b_dev, const void* c_dev, size_t n,
                                             uint8_t* verdict_dev) {
  if (!ctx || !pvk_dev || (n && (!a_dev || !b_dev || !c_dev || !verdict_dev || (m && !inputs_dev))))
    return fail(RIPP_ERR_ARG, "null argument");
  if (n > (size_t)0xffffffffu) return fail(RIPP_ERR_ARG, "more than 2^32 - 1 proofs");
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  return verify_batch(ctx, pvk_dev, m, inputs_dev, a_dev, b_dev, c_dev, n, nullptr, verdict_dev);
}

extern "C" int ripp_groth16_verify_serialized(ripp_ctx* ctx, const void* pvk_dev, size_t m, const uint8_t* inputs_host,
                                              size_t inputs_len, const uint8_t* proofs_host, size_t proofs_len, size_t n,
                                              int compressed, uint8_t* status_host, size_t* n_valid) {
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
  OK(verify_batch(ctx, pvk_dev, m, x, dp.a, dp.b, dp.c, n, st, st));
  CU(cudaMemcpyAsync(status_host, st, n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  size_t ok = 0;
  for (size_t i = 0; i < n; i++) ok += status_host[i] == RIPP_GROTH16_OK;
  *n_valid = ok;
  return RIPP_OK;
}
