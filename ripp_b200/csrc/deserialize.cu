// Validated decoding of ark-serialize point encodings on the GPU, and aggregate_proofs starting from the bytes of the
// Groth16 proofs (include/ripp_b200.h "deserialisation").  Untrusted input: every element is checked -- flags, canonical
// coordinates, curve, prime-order subgroup (serde.cuh) -- before any of it reaches the endomorphism-based kernels of
// the aggregation, whose GLV / GLS maps are scalar multiplications only inside the r-torsion.
#include "common.cuh"
#include "serde.cuh"

// One thread per element: a compressed G2 point costs two Fq exponentiations, an inversion and the subgroup test
// (~3 k Fq products), so the work is throughput-bound from a few thousand elements up.  Small blocks spread a 2^12
// batch over more SMs.
template <bool COMPRESSED>
__global__ void __launch_bounds__(64) k_g1_deserialize(const uint8_t* __restrict__ in, uint32_t n, size_t stride,
                                                       G1Aff* __restrict__ out, uint8_t* __restrict__ status) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  status[i] = serde::decode_point<Fq, COMPRESSED>(in + i * stride, out + i);
}
template <bool COMPRESSED>
__global__ void __launch_bounds__(64) k_g2_deserialize(const uint8_t* __restrict__ in, uint32_t n, size_t stride,
                                                       G2Aff* __restrict__ out, uint8_t* __restrict__ status) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  status[i] = serde::decode_point<Fq2, COMPRESSED>(in + i * stride, out + i);
}

template <class F>
static int deserialize_dev(ripp_ctx* ctx, const void* bytes_dev, size_t n, size_t stride, int compressed, void* out_dev,
                           uint8_t* status_dev) {
  const size_t elem = (compressed ? 48 : 96) * (sizeof(F) / sizeof(Fq));
  if (!ctx || (n && (!bytes_dev || !out_dev || !status_dev))) return fail(RIPP_ERR_ARG, "null argument");
  if (stride < elem)
    return fail(RIPP_ERR_ARG, "stride " + std::to_string(stride) + " is shorter than one encoded element (" + std::to_string(elem) + " bytes)");
  if (n > 0xffffffffu) return fail(RIPP_ERR_ARG, "more than 2^32 - 1 elements");
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  const unsigned nb = (unsigned)((n + 63) / 64);
  const uint8_t* in = (const uint8_t*)bytes_dev;
  if (sizeof(F) == sizeof(Fq)) {
    if (compressed)
      k_g1_deserialize<true><<<nb, 64, 0, ctx->stream>>>(in, (uint32_t)n, stride, (G1Aff*)out_dev, status_dev);
    else
      k_g1_deserialize<false><<<nb, 64, 0, ctx->stream>>>(in, (uint32_t)n, stride, (G1Aff*)out_dev, status_dev);
  } else {
    if (compressed)
      k_g2_deserialize<true><<<nb, 64, 0, ctx->stream>>>(in, (uint32_t)n, stride, (G2Aff*)out_dev, status_dev);
    else
      k_g2_deserialize<false><<<nb, 64, 0, ctx->stream>>>(in, (uint32_t)n, stride, (G2Aff*)out_dev, status_dev);
  }
  LAUNCHED(ctx);
  return RIPP_OK;
}

extern "C" int ripp_g1_deserialize_dev(ripp_ctx* ctx, const void* bytes_dev, size_t n, size_t stride, int compressed,
                                       void* g1_aff_out_dev, uint8_t* status_dev) {
  return deserialize_dev<Fq>(ctx, bytes_dev, n, stride, compressed, g1_aff_out_dev, status_dev);
}
extern "C" int ripp_g2_deserialize_dev(ripp_ctx* ctx, const void* bytes_dev, size_t n, size_t stride, int compressed,
                                       void* g2_aff_out_dev, uint8_t* status_dev) {
  return deserialize_dev<Fq2>(ctx, bytes_dev, n, stride, compressed, g2_aff_out_dev, status_dev);
}

static const char* decode_status_text(uint8_t s) {
  switch (s) {
    case serde::FLAGS: return "has invalid flag bits";
    case serde::NONCANONICAL: return "has a non-canonical coordinate (>= p)";
    case serde::NOT_ON_CURVE: return "not on the curve";
    case serde::NOT_IN_SUBGROUP: return "not in the prime-order subgroup";
  }
  return "invalid";
}

extern "C" int ripp_tipp_aggregate_serialized(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev,
                                              const uint8_t* proofs_host, size_t proofs_len, size_t n, int compressed,
                                              uint8_t* proof_out, size_t proof_cap, size_t* proof_len) {
  if (!ctx || !srs_g1_dev || !srs_g2_dev || !proofs_host) return fail(RIPP_ERR_ARG, "null argument");
  const size_t g1b = compressed ? 48 : 96, g2b = 2 * g1b, rec = 2 * g1b + g2b;
  if (n > (size_t)0xffffffffu || proofs_len != n * rec)
    return fail(RIPP_ERR_ARG, "proof bytes: " + std::to_string(proofs_len) + " bytes is not " + std::to_string(n) + " records of " +
                                  std::to_string(rec) + " bytes");
  if (n == 0 || (n & (n - 1))) return fail(RIPP_ERR_NOT_POW2, "number of proofs must be a power of two");
  if (n < 2) return fail(RIPP_ERR_ARG, "aggregation needs at least two proofs (tipa/mod.rs:199 unwraps the first challenge)");
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  const size_t o_a = up(n * rec), o_b = o_a + n * 96, o_c = o_b + n * 192, o_st = o_c + n * 96;
  void* d;
  OK(scratch(ctx, 23, o_st + up(3 * n), &d));
  char* D = (char*)d;
  uint8_t* S = (uint8_t*)(D + o_st);
  CU(cudaMemcpyAsync(D, proofs_host, n * rec, cudaMemcpyHostToDevice, st));
  // A, B, C on three streams: at 2^12 proofs one component alone does not fill the GPU
  ripp_ctx* kb = ripp_child(ctx, 0);
  ripp_ctx* kc = ripp_child(ctx, 1);
  if (!kb || !kc) return fail(RIPP_ERR_CUDA, "child context");
  OK(ripp_fork(ctx, kb));
  OK(ripp_fork(ctx, kc));
  OK(ripp_g2_deserialize_dev(kb, D + g1b, n, rec, compressed, D + o_b, S + n));
  OK(ripp_g1_deserialize_dev(kc, D + g1b + g2b, n, rec, compressed, D + o_c, S + 2 * n));
  OK(ripp_g1_deserialize_dev(ctx, D, n, rec, compressed, D + o_a, S));
  OK(ripp_join(ctx, kb));
  OK(ripp_join(ctx, kc));
  std::vector<uint8_t> status(3 * n);
  CU(cudaMemcpyAsync(status.data(), S, 3 * n, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  for (size_t i = 0; i < n; i++)
    for (int c = 0; c < 3; c++)
      if (uint8_t s = status[c * n + i])
        return fail(RIPP_ERR_ARG, "proof " + std::to_string(i) + ": " + "ABC"[c] + " " + decode_status_text(s));
  return ripp_tipp_aggregate_dev(ctx, srs_g1_dev, srs_g2_dev, D + o_a, D + o_b, D + o_c, n, proof_out, proof_cap, proof_len);
}
