// Fixed-base windowed scalar multiplication and the setup entry points of the hot path.
//
// Replaces (paths relative to the arkworks-rs/ripp checkout; SURVEY.md §8 rows a9, a14):
//   ip_proofs/src/tipa/mod.rs:372-391   structured_generators_scalar_power (ark-ec FixedBase::get_window_table / msm)
//   ip_proofs/src/tipa/mod.rs:150-164   TIPA::setup -- the SRS { g^(alpha^i), h^(beta^i), g^beta, h^alpha }
//   dh_commitments/src/lib.rs:59-61     random_generators, behind AFGHO16 / Pedersen `setup`
//     (afgho16/mod.rs:36-38,58-60; pedersen/mod.rs:20-22)
// The random draws themselves (Fr::rand / G::rand on the caller's RNG) stay with the caller: the entry points take
// the trapdoors / exponents, so the reference's random stream is the reference's own (INTEGRATION.md "setup").
//
// Shape: one table of (2^c - 1) * ceil(255 / c) affine multiples d 2^(c w) B of the base, built by ONE launch of the
// element-wise scaling kernel on the table's exponents (no serial doubling chain), then one thread per output adds
// its ceil(255 / c) table entries (mixed additions) and normalises.  c = 8: 8160 entries (0.8 MB in G1, 1.6 MB in
// G2: L2 resident), 32 additions per output against ~255 doublings + ~85 additions of the variable-base path.
#include "common.cuh"

constexpr int FB_C = 8;
constexpr int FB_NW = (255 + FB_C - 1) / FB_C;
constexpr int FB_PER = (1 << FB_C) - 1;

constexpr int FB_ENTRIES = FB_NW * FB_PER;

// exponents of the tables: t[b * FB_ENTRIES + w * FB_PER + d - 1] = d 2^(c w) (Montgomery), b < nb; with the bases
// (non-null) repeated alongside, pts[b * FB_ENTRIES + e] = bases[b], so that one scaling launch builds nb tables
__global__ void k_fb_exponents(Fr* __restrict__ t, int nb, const G1Aff* __restrict__ bases, G1Aff* __restrict__ pts) {
  int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= nb * FB_ENTRIES) return;
  if (bases) pts[g] = bases[g / FB_ENTRIES];
  int e = g % FB_ENTRIES, w = e / FB_PER, d = e % FB_PER + 1;
  Fr v = Fr::zero();
  v.v[0] = (uint32_t)d;
  v = v.to_mont();
  for (int i = 0; i < FB_C * w; i++) v = v.dbl();
  t[g] = v;
}

// acc += s B, s Montgomery, from the table of B: one mixed addition per 8-bit window
template <class F>
__device__ __forceinline__ Jac<F> fb_add(Jac<F> acc, const Aff<F>* __restrict__ table, const Fr& sc) {
  Fr s = sc.from_mont();
  for (int w = 0; w < FB_NW; w++) {
    int o = w * FB_C, wi = o >> 5, sh = o & 31;
    uint64_t v = s.v[wi];
    if (wi + 1 < 8) v |= (uint64_t)s.v[wi + 1] << 32;
    uint32_t d = (uint32_t)(v >> sh) & FB_PER;
    Aff<F> q = d ? table[w * FB_PER + d - 1] : Aff<F>::inf();  // digit 0 adds the identity: same instruction stream
    acc = Jac<F>::add_mixed_fn(acc, q);
  }
  return acc;
}

template <class F>
__global__ void __launch_bounds__(64, 4) k_fb_msm(const Aff<F>* __restrict__ table, const Fr* __restrict__ sc, size_t n,
                                               Aff<F>* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  out[i] = fb_add<F>(Jac<F>::inf(), table, sc[i]).to_affine();
}

// Groth16 prepare_inputs for n proofs: P_i = IC_0 + sum_j x_ij IC_(j+1) over the m tables of IC_1..IC_m
// (groth16.cu); one thread per proof, m x 32 mixed additions
__global__ void __launch_bounds__(64, 4) k_groth16_inputs(const G1Aff* __restrict__ ic0, const G1Aff* __restrict__ tables,
                                                       const Fr* __restrict__ x, uint32_t n, uint32_t m, G1Aff* __restrict__ out) {
  uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Jac<Fq> acc = Jac<Fq>::from_affine(*ic0);
  for (uint32_t j = 0; j < m; j++) acc = fb_add<Fq>(acc, tables + (size_t)j * FB_ENTRIES, x[(size_t)i * m + j]);
  out[i] = acc.to_affine();
}

// s^i, i < n, by square-and-multiply on the index
__global__ void k_fr_power_seq(Fr s, size_t n, Fr* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Fr acc = Fr::one(), b = s;
  for (size_t e = i; e; e >>= 1) {
    if (e & 1) acc = acc * b;
    b = b * b;
  }
  out[i] = acc;
}
int ripp_fr_power_seq_internal(ripp_ctx* ctx, const Fr& s, size_t n, void* out_dev) {
  if (n == 0) return RIPP_OK;
  k_fr_power_seq<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>(s, n, (Fr*)out_dev);
  LAUNCHED(ctx);
  return RIPP_OK;
}

int ripp_scale_base_g1(ripp_ctx* ctx, const G1Aff* base_or_null, const void* sc_dev, size_t n, void* out_dev);
int ripp_scale_base_g2(ripp_ctx* ctx, const G2Aff* base_or_null, const void* sc_dev, size_t n, void* out_dev);

// The fixed-base tables of nb bases (FB_ENTRIES affine points each, written to `tables`): one exponent launch and ONE
// scaling launch for all of them.  Either one base (host, or NULL for the generator), or nb G1 bases in device memory.
template <class F>
static int fb_tables(ripp_ctx* ctx, const Aff<F>* base_host, const G1Aff* bases_dev, size_t nb, Aff<F>* tables) {
  const size_t ne = nb * FB_ENTRIES, o_pts = (ne * sizeof(Fr) + 255) & ~(size_t)255;
  void* buf;
  OK(scratch(ctx, 31, o_pts + (bases_dev ? ne * sizeof(G1Aff) : 0), &buf));
  Fr* ex = (Fr*)buf;
  G1Aff* pts = bases_dev ? (G1Aff*)((char*)buf + o_pts) : nullptr;
  k_fb_exponents<<<(unsigned)((ne + 127) / 128), 128, 0, ctx->stream>>>(ex, (int)nb, bases_dev, pts);
  LAUNCHED(ctx);
  if (bases_dev) return ripp_g1_scale_dev(ctx, pts, ex, ne, tables);
  if (sizeof(F) == sizeof(Fq)) return ripp_scale_base_g1(ctx, (const G1Aff*)base_host, ex, ne, tables);
  return ripp_scale_base_g2(ctx, (const G2Aff*)base_host, ex, ne, tables);
}

template <class F>
static int fixed_base_msm(ripp_ctx* ctx, const void* base_host, const void* sc_dev, size_t n, void* out_dev) {
  if (!ctx || (n && (!sc_dev || !out_dev))) return fail(RIPP_ERR_ARG, "null argument");
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  Aff<F> base;
  if (base_host) memcpy(&base, base_host, sizeof(base));
  // short vectors: the table (8160 scalar multiplications) would cost more than the outputs
  if (n < 2048) {
    if (sizeof(F) == sizeof(Fq)) return ripp_scale_base_g1(ctx, base_host ? (const G1Aff*)&base : nullptr, sc_dev, n, out_dev);
    return ripp_scale_base_g2(ctx, base_host ? (const G2Aff*)&base : nullptr, sc_dev, n, out_dev);
  }
  void* buf;
  OK(scratch(ctx, 24, (size_t)FB_ENTRIES * sizeof(Aff<F>), &buf));
  Aff<F>* table = (Aff<F>*)buf;
  OK(fb_tables<F>(ctx, base_host ? &base : nullptr, nullptr, 1, table));
  TimeScope ts_(ctx, RIPP_T_SCALE);
  k_fb_msm<F><<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>(table, (const Fr*)sc_dev, n, (Aff<F>*)out_dev);
  LAUNCHED(ctx);
  return RIPP_OK;
}

extern "C" int ripp_fixed_base_msm_g1_dev(ripp_ctx* ctx, const void* base_g1_aff, const void* fr_dev, size_t n, void* out_dev) {
  return fixed_base_msm<Fq>(ctx, base_g1_aff, fr_dev, n, out_dev);
}
extern "C" int ripp_fixed_base_msm_g2_dev(ripp_ctx* ctx, const void* base_g2_aff, const void* fr_dev, size_t n, void* out_dev) {
  return fixed_base_msm<Fq2>(ctx, base_g2_aff, fr_dev, n, out_dev);
}

template <class F>
static int structured_generators(ripp_ctx* ctx, const void* base_host, const void* s_host, size_t num, void* out_dev) {
  if (!ctx || !s_host || !out_dev) return fail(RIPP_ERR_ARG, "null argument");
  if (num == 0) return fail(RIPP_ERR_ARG, "structured_generators_scalar_power: num must be positive (tipa/mod.rs:377)");
  CU(cudaSetDevice(ctx->device));
  Fr s;
  memcpy(s.v, s_host, sizeof(Fr));
  void* pw;
  OK(scratch(ctx, 25, num * sizeof(Fr) + 256, &pw));
  OK(ripp_fr_power_seq_internal(ctx, s, num, pw));
  return fixed_base_msm<F>(ctx, base_host, pw, num, out_dev);
}
extern "C" int ripp_structured_generators_g1_dev(ripp_ctx* ctx, const void* base_g1_aff, const void* s, size_t num, void* out_dev) {
  return structured_generators<Fq>(ctx, base_g1_aff, s, num, out_dev);
}
extern "C" int ripp_structured_generators_g2_dev(ripp_ctx* ctx, const void* base_g2_aff, const void* s, size_t num, void* out_dev) {
  return structured_generators<Fq2>(ctx, base_g2_aff, s, num, out_dev);
}

extern "C" int ripp_tipa_setup_dev(ripp_ctx* ctx, const void* alpha, const void* beta, size_t size, void* srs_g1_out_dev,
                                   void* srs_g2_out_dev, void* g_beta_out, void* h_alpha_out) {
  if (!ctx || !alpha || !beta || !srs_g1_out_dev || !srs_g2_out_dev || !g_beta_out || !h_alpha_out)
    return fail(RIPP_ERR_ARG, "null argument");
  if (size == 0) return fail(RIPP_ERR_ARG, "TIPA::setup: size must be positive");
  CU(cudaSetDevice(ctx->device));
  const size_t m = 2 * size - 1;
  // the two towers of powers run on two streams
  ripp_ctx* kid = ripp_child(ctx, 0);
  if (!kid) return fail(RIPP_ERR_CUDA, "child context");
  OK(ripp_fork(ctx, kid));
  OK(structured_generators<Fq2>(kid, nullptr, beta, m, srs_g2_out_dev));
  OK(structured_generators<Fq>(ctx, nullptr, alpha, m, srs_g1_out_dev));
  OK(ripp_join(ctx, kid));
  // g^beta, h^alpha
  void* d;
  OK(scratch(ctx, 26, 1024, &d));
  char* p = (char*)d;
  CU(cudaMemcpyAsync(p, beta, 32, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(p + 32, alpha, 32, cudaMemcpyHostToDevice, ctx->stream));
  OK(ripp_scale_base_g1(ctx, nullptr, p, 1, p + 256));
  OK(ripp_scale_base_g2(ctx, nullptr, p + 32, 1, p + 512));
  CU(cudaMemcpyAsync(g_beta_out, p + 256, 96, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaMemcpyAsync(h_alpha_out, p + 512, 192, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

// ---- Groth16 prepare_inputs (groth16.cu) -------------------------------------------------------------------------
size_t ripp_groth16_table_bytes() { return (size_t)FB_ENTRIES * sizeof(G1Aff); }

int ripp_groth16_tables(ripp_ctx* ctx, const void* ic_dev, size_t m, void* tables_dev) {
  if (m == 0) return RIPP_OK;
  return fb_tables<Fq>(ctx, nullptr, (const G1Aff*)ic_dev, m, (G1Aff*)tables_dev);
}

int ripp_groth16_inputs(ripp_ctx* ctx, const void* ic0_dev, const void* tables_dev, size_t m, const void* x_dev, size_t n,
                        void* out_dev) {
  TimeScope ts_(ctx, RIPP_T_SCALE);
  k_groth16_inputs<<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>((const G1Aff*)ic0_dev, (const G1Aff*)tables_dev,
                                                                      (const Fr*)x_dev, (uint32_t)n, (uint32_t)m, (G1Aff*)out_dev);
  LAUNCHED(ctx);
  return RIPP_OK;
}
