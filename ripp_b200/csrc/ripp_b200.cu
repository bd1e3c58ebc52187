// ripp_b200: CUDA kernels (sm_100a) + C ABI (include/ripp_b200.h).
#include "common.cuh"
#include "x3.cuh"
#include "endo.cuh"
#include "xt.cuh"

static thread_local std::string g_err;
std::string& ripp_err_slot() { return g_err; }

extern "C" const char* ripp_last_error_string(void) { return g_err.c_str(); }

extern "C" int ripp_ctx_create(int device, ripp_ctx** out) {
  if (!out) return fail(RIPP_ERR_ARG, "null out");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0)
    return fail(RIPP_ERR_NO_DEVICE, std::string("no CUDA device (ripp_b200 has no CPU fallback): ") + cudaGetErrorString(e));
  if (device < 0 || device >= count) return fail(RIPP_ERR_ARG, "bad device ordinal");
  CU(cudaSetDevice(device));
  OK(ripp_pairing6_init_device());
  ripp_ctx* c = new ripp_ctx();
  memset(c, 0, sizeof(*c));
  c->device = device;
  c->world = 1;
  CU(cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
  c->stream = c->own_stream;
  c->recs = new std::vector<TimingRec>();
  CU(cudaEventCreateWithFlags(&c->ev, cudaEventDisableTiming));
  *out = c;
  return RIPP_OK;
}

ripp_ctx* ripp_child(ripp_ctx* ctx, int idx) {
  if (idx < 0 || idx >= RIPP_MAX_CHILD) return nullptr;
  if (!ctx->child[idx]) {
    ripp_ctx* c = nullptr;
    if (ripp_ctx_create(ctx->device, &c) != RIPP_OK) return nullptr;
    c->parent = ctx;
    ctx->child[idx] = c;
  }
  ctx->child[idx]->timing = ctx->timing;
  return ctx->child[idx];
}
int ripp_fork(ripp_ctx* ctx, ripp_ctx* child) {
  CU(cudaEventRecord(ctx->ev, ctx->stream));
  CU(cudaStreamWaitEvent(child->stream, ctx->ev, 0));
  return RIPP_OK;
}
int ripp_join(ripp_ctx* ctx, ripp_ctx* child) {
  CU(cudaEventRecord(child->ev, child->stream));
  CU(cudaStreamWaitEvent(ctx->stream, child->ev, 0));
  return RIPP_OK;
}

extern "C" void ripp_ctx_destroy(ripp_ctx* ctx) {
  if (!ctx) return;
  cudaSetDevice(ctx->device);
  cudaStreamSynchronize(ctx->stream);
  for (int i = 0; i < RIPP_MAX_CHILD; i++)
    if (ctx->child[i]) ripp_ctx_destroy(ctx->child[i]);
  ripp_comm_release(ctx);
  cudaEventDestroy(ctx->ev);
  for (int i = 0; i < RIPP_SCRATCH_SLOTS; i++)
    if (ctx->scratch[i]) cudaFree(ctx->scratch[i]);
  cudaStreamDestroy(ctx->own_stream);
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  if (ctx->pinned_big) cudaFreeHost(ctx->pinned_big);
  if (ctx->recs) {
    for (auto& r : *ctx->recs) {
      cudaEventDestroy(r.a);
      cudaEventDestroy(r.b);
    }
    delete ctx->recs;
  }
  delete ctx;
}

extern "C" int ripp_ctx_sync(ripp_ctx* ctx) {
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}
extern "C" void* ripp_ctx_stream(ripp_ctx* ctx) { return (void*)ctx->stream; }
extern "C" int ripp_ctx_set_stream(ripp_ctx* ctx, void* s) {
  if (!ctx) return fail(RIPP_ERR_ARG, "null ctx");
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
  return RIPP_OK;
}
extern "C" uint64_t ripp_ctx_launch_count(ripp_ctx* ctx) {
  uint64_t n = ctx->launches;
  for (int i = 0; i < RIPP_MAX_CHILD; i++)
    if (ctx->child[i]) n += ripp_ctx_launch_count(ctx->child[i]);
  return n;
}
extern "C" int ripp_ctx_set_timing(ripp_ctx* ctx, int on) {
  if (!ctx) return fail(RIPP_ERR_ARG, "null ctx");
  ctx->timing = on;
  return RIPP_OK;
}
static int timing_collect(ripp_ctx* ctx, double* ms_by_cat, uint64_t* count_by_cat) {
  CU(cudaStreamSynchronize(ctx->stream));
  for (int i = 0; i < RIPP_MAX_CHILD; i++)
    if (ctx->child[i]) OK(timing_collect(ctx->child[i], ms_by_cat, count_by_cat));
  for (auto& r : *ctx->recs) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      ms_by_cat[r.cat] += ms;
      count_by_cat[r.cat]++;
    }
    cudaEventDestroy(r.a);
    cudaEventDestroy(r.b);
  }
  ctx->recs->clear();
  return RIPP_OK;
}
extern "C" int ripp_ctx_timing(ripp_ctx* ctx, double* ms_by_cat, uint64_t* count_by_cat) {
  if (!ctx || !ms_by_cat || !count_by_cat) return fail(RIPP_ERR_ARG, "null argument");
  for (int i = 0; i < RIPP_T_NCAT; i++) {
    ms_by_cat[i] = 0;
    count_by_cat[i] = 0;
  }
  return timing_collect(ctx, ms_by_cat, count_by_cat);
}

extern "C" int ripp_dev_alloc(ripp_ctx* ctx, size_t bytes, void** dev_out) {
  CU(cudaSetDevice(ctx->device));
  CU(cudaMalloc(dev_out, bytes ? bytes : 16));
  return RIPP_OK;
}
extern "C" int ripp_dev_free(ripp_ctx* ctx, void* dev) {
  CU(cudaSetDevice(ctx->device));
  CU(cudaStreamSynchronize(ctx->stream));
  CU(cudaFree(dev));
  return RIPP_OK;
}
extern "C" int ripp_dev_upload(ripp_ctx* ctx, void* dev_dst, const void* host_src, size_t bytes) {
  CU(cudaMemcpyAsync(dev_dst, host_src, bytes, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}
extern "C" int ripp_dev_download(ripp_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes) {
  CU(cudaMemcpyAsync(host_dst, dev_src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

// ------------------------------------------------------------------------------------------------
// kernels: normalisation (inner_products/src/lib.rs:80-81 normalize_batch)
// ------------------------------------------------------------------------------------------------
template <class F>
__global__ void k_normalize(const Jac<F>* __restrict__ in, Aff<F>* __restrict__ out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Jac<F> p = in[i];
  Aff<F> a;
  if (p.is_inf())
    a = Aff<F>::inf();
  else if (p.z == F::one())
    a = {p.x, p.y};
  else
    a = p.to_affine();
  out[i] = a;
}

// ------------------------------------------------------------------------------------------------
// kernels: element-wise scalar multiplication with distinct scalars (K8)
// ------------------------------------------------------------------------------------------------
template <class F, bool GEN>
__global__ void __launch_bounds__(64, 4) k_scale(const Aff<F>* __restrict__ pts, const Fr* __restrict__ sc, size_t n,
                                              Aff<F>* __restrict__ out, Aff<F> gen) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  // every lane stays alive for the full-mask shuffles below: lanes past n redo element n - 1 and do not store
  const bool live = i < n;
  if (!live) i = n - 1;
  Fr s = sc[i].from_mont();
  Aff<F> p = GEN ? gen : pts[i];
  EndoBits eb;  // GLV / GLS decomposition of this element's scalar (endo.cuh)
  endo_decompose<sizeof(F) == sizeof(Fq) ? 1 : 2>(s.v, eb);
  // warp-uniform trip counts (every lane walks the longest digit of the warp)
  int nb = eb.nbits, mm = eb.m;
  for (int o = 16; o >= 1; o >>= 1) {
    nb = max(nb, __shfl_xor_sync(0xffffffffu, nb, o));
    mm = max(mm, __shfl_xor_sync(0xffffffffu, mm, o));
  }
  nb = min(nb, 160);  // bounds of EndoBits::pos / neg and base[4], whatever the decomposition returned
  mm = min(mm, 4);
  Aff<F> r = endo_mul_simt<F>(p, eb, mm, nb).to_affine();
  if (live) out[i] = r;
}

// Short vectors (the 2^12-element scalings a_i r^i / ck_i r^-i of aggregate_proofs were 4096 lone threads, 10.7 ms for G2):
// one thread per (element, endomorphism part).  s P = sum_t d_t E^t(P) (endo.cuh) is m independent scalar
// multiplications with 128-bit (G1, m = 2) / 64-bit (G2, m = 4) scalars: m times the parallelism at 1/m of the chain,
// then one thread per element adds the m parts and normalises.  Lane teams (k_scale_xt below, kept for A/B runs) were
// measured SLOWER here (8.8 ms): at 1366 warps the redundant glue of nine lanes per element is throughput, not latency.
// So were three-WARP teams per 32 (element, part) chains (x3.cuh, G2: 4.96 ms against 4.06 ms, gpurun_out r2j): the CTA
// barriers of ~1150 exchanges and 2.4 KB of spills cost more than the shorter chain returns.
template <class F, bool GEN>
__global__ void __launch_bounds__(64, 4) k_scale_parts(const Aff<F>* __restrict__ pts, const Fr* __restrict__ sc, size_t n, int m,
                                                    Jac<F>* __restrict__ parts, Aff<F> gen) {
  size_t g = (size_t)blockIdx.x * blockDim.x + threadIdx.x;  // g = t n + i: a warp works on one part index (mostly)
  const bool live = g < (size_t)m * n;
  if (!live) g = (size_t)m * n - 1;
  const int t = (int)(g / n);
  const size_t i = g % n;
  Fr s = sc[i].from_mont();
  uint32_t digits[4][4];
  int mm;
  endo_digits<sizeof(F) == sizeof(Fq) ? 1 : 2>(s.v, digits, &mm);
  Aff<F> p = GEN ? gen : pts[i];
  {  // E^t(P): the chain of images as endo_mul_simt forms it, then a select (no data-dependent trip count)
    Aff<F> b1 = endo_map(p), b2 = endo_map(b1), b3 = endo_map(b2);
    p = t == 0 ? p : (t == 1 ? b1 : (t == 2 ? b2 : b3));
  }
  uint32_t d[4], pos[5] = {0, 0, 0, 0, 0}, neg[5] = {0, 0, 0, 0, 0};
  for (int j = 0; j < 4; j++) d[j] = t == 0 ? digits[0][j] : (t == 1 ? digits[1][j] : (t == 2 ? digits[2][j] : digits[3][j]));
  int nd = 0;
  naf_bitmaps(d, 4, pos, neg, &nd);
  for (int o = 16; o >= 1; o >>= 1) nd = max(nd, __shfl_xor_sync(0xffffffffu, nd, o));
  nd = min(nd, 160);
  const Aff<F> np = p.neg();
  Jac<F> acc = Jac<F>::inf();
  for (int j = nd - 1; j >= 0; j--) {
    acc = Jac<F>::dbl_fn(acc);
    const bool ps = (pos[j >> 5] >> (j & 31)) & 1, ng = (neg[j >> 5] >> (j & 31)) & 1;
    Aff<F> q = ng ? np : p;
    if (!(ps || ng)) q = Aff<F>::inf();
    acc = Jac<F>::add_mixed_fn(acc, q);
  }
  if (live) parts[g] = acc;
}
template <class F>
__global__ void __launch_bounds__(64, 4) k_scale_combine(const Jac<F>* __restrict__ parts, size_t n, int m, Aff<F>* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Jac<F> acc = parts[i];
  for (int t = 1; t < m; t++) acc = acc.add(parts[(size_t)t * n + i]);
  out[i] = acc.to_affine();
}
static size_t scale_parts_max_n() {
  static const long v = [] {
    const char* e = getenv("RIPP_B200_SCALE_PARTS_MAX");  // 0 = one thread per element everywhere (A/B runs)
    return e ? atol(e) : 16384L;
  }();
  return (size_t)v;
}

// Lane teams (xt.cuh: 3 lanes per G1 element, 9 per G2 element) for vectors short enough that one element's dependent
// chain, not the multiplier pipe, is the cost: the 2^12-element scalings of aggregate_proofs were 4096 lone threads.
constexpr int SXT_WARPS = 2;
template <class F, bool GEN>
__global__ void __launch_bounds__(32 * SXT_WARPS) k_scale_xt(const Aff<F>* __restrict__ pts, const Fr* __restrict__ sc, size_t n,
                                                            Aff<F>* __restrict__ out, Aff<F> gen) {
  typedef xt::TeamOf<F> TO;
  constexpr int AW4 = 4 * sizeof(Aff<F>) / 4;
  __shared__ __align__(16) uint32_t bus[SXT_WARPS * TO::PER_WARP * (2 * TO::BUS_WORDS + AW4)];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int vl = lane % (TO::LANES * TO::PER_WARP);
  const int e = vl / TO::LANES;
  size_t i = ((size_t)blockIdx.x * SXT_WARPS + warp) * TO::PER_WARP + e;
  const bool live = i < n && lane == vl;
  if (i >= n) i = n - 1;
  uint32_t* scratch = bus + (warp * TO::PER_WARP + e) * (2 * TO::BUS_WORDS + AW4);
  xt::Team tm{vl % TO::LANES, scratch, 0, nullptr};
  Fr s = sc[i].from_mont();
  EndoBits eb;
  endo_decompose<sizeof(F) == sizeof(Fq) ? 1 : 2>(s.v, eb);
  int nb = eb.nbits, mm = eb.m;
  for (int o = 16; o >= 1; o >>= 1) {
    nb = max(nb, __shfl_xor_sync(0xffffffffu, nb, o));
    mm = max(mm, __shfl_xor_sync(0xffffffffu, mm, o));
  }
  nb = min(nb, 160);
  mm = min(mm, 4);
  Jac<F> acc = xt::endo_mul_sel<F>(tm, GEN ? gen : pts[i], eb, mm, nb, scratch + 2 * TO::BUS_WORDS);
  Aff<F> o = xt::to_affine<F>(tm, acc);
  if (live && tm.t == 0) out[i] = o;
}
static size_t scale_xt_max_n(bool g2) {
  static const long v = [] {
    const char* e = getenv("RIPP_B200_SCALE_XT_MAX");  // 0 = one thread per element everywhere (A/B runs)
    return e ? atol(e) : -1L;
  }();
  return v >= 0 ? (size_t)v : 0;  // off by default: see k_scale_parts
}

template <class F, class XF>
static int scale_dev(ripp_ctx* ctx, const void* pts, const void* sc, size_t n, void* out, const Aff<F>& gen) {
  if (!ctx || (n && (!sc || !out))) return fail(RIPP_ERR_ARG, "null argument");
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  TimeScope ts_(ctx, RIPP_T_SCALE);
  if (n <= scale_parts_max_n()) {
    const int m = sizeof(F) == sizeof(Fq) ? 2 : 4;
    void* parts;
    OK(scratch(ctx, 22, (size_t)m * n * sizeof(Jac<F>), &parts));
    unsigned blocks = (unsigned)(((size_t)m * n + 63) / 64);
    if (pts)
      k_scale_parts<F, false><<<blocks, 64, 0, ctx->stream>>>((const Aff<F>*)pts, (const Fr*)sc, n, m, (Jac<F>*)parts, gen);
    else
      k_scale_parts<F, true><<<blocks, 64, 0, ctx->stream>>>(nullptr, (const Fr*)sc, n, m, (Jac<F>*)parts, gen);
    LAUNCHED(ctx);
    k_scale_combine<F><<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>((const Jac<F>*)parts, n, m, (Aff<F>*)out);
    LAUNCHED(ctx);
    return RIPP_OK;
  }
  if (n <= scale_xt_max_n(sizeof(F) != sizeof(Fq))) {
    typedef xt::TeamOf<F> TO;
    unsigned warps = (unsigned)((n + TO::PER_WARP - 1) / TO::PER_WARP), blocks = (warps + SXT_WARPS - 1) / SXT_WARPS;
    if (pts)
      k_scale_xt<F, false><<<blocks, 32 * SXT_WARPS, 0, ctx->stream>>>((const Aff<F>*)pts, (const Fr*)sc, n, (Aff<F>*)out, gen);
    else
      k_scale_xt<F, true><<<blocks, 32 * SXT_WARPS, 0, ctx->stream>>>(nullptr, (const Fr*)sc, n, (Aff<F>*)out, gen);
    LAUNCHED(ctx);
    return RIPP_OK;
  }
  unsigned blocks = (unsigned)((n + 63) / 64);
  if (pts)
    k_scale<F, false><<<blocks, 64, 0, ctx->stream>>>((const Aff<F>*)pts, (const Fr*)sc, n, (Aff<F>*)out, gen);
  else
    k_scale<F, true><<<blocks, 64, 0, ctx->stream>>>(nullptr, (const Fr*)sc, n, (Aff<F>*)out, gen);
  LAUNCHED(ctx);
  return RIPP_OK;
}
// the same kernels on one caller-supplied base (setup.cu: the fixed-base table and the short-vector path)
int ripp_scale_base_g1(ripp_ctx* ctx, const G1Aff* base_or_null, const void* sc, size_t n, void* out) {
  return scale_dev<Fq, Fq>(ctx, nullptr, sc, n, out, base_or_null ? *base_or_null : g1_generator());
}
int ripp_scale_base_g2(ripp_ctx* ctx, const G2Aff* base_or_null, const void* sc, size_t n, void* out) {
  return scale_dev<Fq2, x3::Fq2x3>(ctx, nullptr, sc, n, out, base_or_null ? *base_or_null : g2_generator());
}
extern "C" int ripp_g1_scale_dev(ripp_ctx* ctx, const void* pts, const void* sc, size_t n, void* out) {
  return scale_dev<Fq, Fq>(ctx, pts, sc, n, out, g1_generator());
}
extern "C" int ripp_g2_scale_dev(ripp_ctx* ctx, const void* pts, const void* sc, size_t n, void* out) {
  return scale_dev<Fq2, x3::Fq2x3>(ctx, pts, sc, n, out, g2_generator());
}

// ------------------------------------------------------------------------------------------------
// diagnostics
// ------------------------------------------------------------------------------------------------
template <class TA, class TB, class TR, class Fn>
__global__ void k_elementwise(const TA* a, const TB* b, TR* r, size_t n, Fn fn) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) r[i] = fn(a[i], b[i]);
}

template <class TA, class TB, class TR, class Fn>
static int run_elementwise(ripp_ctx* ctx, const void* a, const void* b, void* r, size_t n, Fn fn) {
  void *da, *db, *dr;
  OK(scratch(ctx, 0, n * sizeof(TA), &da));
  OK(scratch(ctx, 1, n * sizeof(TB), &db));
  OK(scratch(ctx, 2, n * sizeof(TR), &dr));
  CU(cudaMemcpyAsync(da, a, n * sizeof(TA), cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(db, b ? b : a, n * (b ? sizeof(TB) : (sizeof(TA) < sizeof(TB) ? sizeof(TA) : sizeof(TB))),
                     cudaMemcpyHostToDevice, ctx->stream));
  int block = 64;
  k_elementwise<TA, TB, TR, Fn><<<(unsigned)((n + block - 1) / block), block, 0, ctx->stream>>>(
      (const TA*)da, (const TB*)db, (TR*)dr, n, fn);
  LAUNCHED(ctx);
  CU(cudaMemcpyAsync(r, dr, n * sizeof(TR), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

struct OpFqMul { __device__ Fq operator()(const Fq& a, const Fq& b) const { return a * b; } };
struct OpFqAdd { __device__ Fq operator()(const Fq& a, const Fq& b) const { return a + b; } };
struct OpFqSub { __device__ Fq operator()(const Fq& a, const Fq& b) const { return a - b; } };
struct OpFqInv { __device__ Fq operator()(const Fq& a, const Fq&) const { return a.inv(); } };
struct OpFqHalf { __device__ Fq operator()(const Fq& a, const Fq&) const { return a.half(); } };
struct OpFrMul { __device__ Fr operator()(const Fr& a, const Fr& b) const { return a * b; } };
struct OpFrAdd { __device__ Fr operator()(const Fr& a, const Fr& b) const { return a + b; } };
struct OpFrSub { __device__ Fr operator()(const Fr& a, const Fr& b) const { return a - b; } };
struct OpFrInv { __device__ Fr operator()(const Fr& a, const Fr&) const { return a.inv(); } };
struct OpFq2Mul { __device__ Fq2 operator()(const Fq2& a, const Fq2& b) const { return a * b; } };
struct OpFq2Sqr { __device__ Fq2 operator()(const Fq2& a, const Fq2&) const { return a.sqr(); } };
struct OpFq2Inv { __device__ Fq2 operator()(const Fq2& a, const Fq2&) const { return a.inv(); } };
struct OpFq12Mul { __device__ Fq12 operator()(const Fq12& a, const Fq12& b) const { return a * b; } };
struct OpFq12Sqr { __device__ Fq12 operator()(const Fq12& a, const Fq12&) const { return a.sqr(); } };
struct OpFq12Inv { __device__ Fq12 operator()(const Fq12& a, const Fq12&) const { return a.inv(); } };
struct OpFq12Cyc { __device__ Fq12 operator()(const Fq12& a, const Fq12&) const { return a.cyclotomic_sqr(); } };
struct OpFq12Frob1 { __device__ Fq12 operator()(const Fq12& a, const Fq12&) const { return a.frob<1>(); } };
struct OpFinalExp { __device__ Fq12 operator()(const Fq12& a, const Fq12&) const { return final_exponentiation(a); } };
struct OpMiller { __device__ Fq12 operator()(const G1Aff& a, const G2Aff& b) const { return miller_loop(a, b); } };
template <class F>
struct OpAdd {
  __device__ Aff<F> operator()(const Aff<F>& a, const Aff<F>& b) const {
    return Jac<F>::from_affine(a).add(Jac<F>::from_affine(b)).to_affine();
  }
};
template <class F>
struct OpDbl {
  __device__ Aff<F> operator()(const Aff<F>& a, const Aff<F>&) const { return Jac<F>::from_affine(a).dbl().to_affine(); }
};

extern "C" int ripp_test_elementwise(ripp_ctx* ctx, int op, const void* a, const void* b, void* r, size_t n) {
  if (!ctx || !a || !r) return fail(RIPP_ERR_ARG, "null argument");
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  switch (op) {
    case RIPP_OP_FQ_MUL: return run_elementwise<Fq, Fq, Fq>(ctx, a, b, r, n, OpFqMul());
    case RIPP_OP_FQ_ADD: return run_elementwise<Fq, Fq, Fq>(ctx, a, b, r, n, OpFqAdd());
    case RIPP_OP_FQ_SUB: return run_elementwise<Fq, Fq, Fq>(ctx, a, b, r, n, OpFqSub());
    case RIPP_OP_FQ_INV: return run_elementwise<Fq, Fq, Fq>(ctx, a, b, r, n, OpFqInv());
    case RIPP_OP_FQ_HALF: return run_elementwise<Fq, Fq, Fq>(ctx, a, b, r, n, OpFqHalf());
    case RIPP_OP_FR_MUL: return run_elementwise<Fr, Fr, Fr>(ctx, a, b, r, n, OpFrMul());
    case RIPP_OP_FR_ADD: return run_elementwise<Fr, Fr, Fr>(ctx, a, b, r, n, OpFrAdd());
    case RIPP_OP_FR_SUB: return run_elementwise<Fr, Fr, Fr>(ctx, a, b, r, n, OpFrSub());
    case RIPP_OP_FR_INV: return run_elementwise<Fr, Fr, Fr>(ctx, a, b, r, n, OpFrInv());
    case RIPP_OP_FQ2_MUL: return run_elementwise<Fq2, Fq2, Fq2>(ctx, a, b, r, n, OpFq2Mul());
    case RIPP_OP_FQ2_SQR: return run_elementwise<Fq2, Fq2, Fq2>(ctx, a, b, r, n, OpFq2Sqr());
    case RIPP_OP_FQ2_INV: return run_elementwise<Fq2, Fq2, Fq2>(ctx, a, b, r, n, OpFq2Inv());
    case RIPP_OP_FQ12_MUL: return run_elementwise<Fq12, Fq12, Fq12>(ctx, a, b, r, n, OpFq12Mul());
    case RIPP_OP_FQ12_SQR: return run_elementwise<Fq12, Fq12, Fq12>(ctx, a, b, r, n, OpFq12Sqr());
    case RIPP_OP_FQ12_INV: return run_elementwise<Fq12, Fq12, Fq12>(ctx, a, b, r, n, OpFq12Inv());
    case RIPP_OP_FQ12_CYC_SQR: return run_elementwise<Fq12, Fq12, Fq12>(ctx, a, b, r, n, OpFq12Cyc());
    case RIPP_OP_FQ12_FROB1: return run_elementwise<Fq12, Fq12, Fq12>(ctx, a, b, r, n, OpFq12Frob1());
    case RIPP_OP_FINAL_EXP: return run_elementwise<Fq12, Fq12, Fq12>(ctx, a, b, r, n, OpFinalExp());
    case RIPP_OP_MILLER: return run_elementwise<G1Aff, G2Aff, Fq12>(ctx, a, b, r, n, OpMiller());
    case RIPP_OP_G1_ADD: return run_elementwise<G1Aff, G1Aff, G1Aff>(ctx, a, b, r, n, OpAdd<Fq>());
    case RIPP_OP_G1_DBL: return run_elementwise<G1Aff, G1Aff, G1Aff>(ctx, a, b, r, n, OpDbl<Fq>());
    case RIPP_OP_G2_ADD: return run_elementwise<G2Aff, G2Aff, G2Aff>(ctx, a, b, r, n, OpAdd<Fq2>());
    case RIPP_OP_G2_DBL: return run_elementwise<G2Aff, G2Aff, G2Aff>(ctx, a, b, r, n, OpDbl<Fq2>());
  }
  return fail(RIPP_ERR_ARG, "unknown test op");
}

// Integer-pipe peak microbenchmark.  8 independent accumulators per thread, register-only.
template <int KIND>
__global__ void __launch_bounds__(256) k_imad(uint32_t* out, int iters, uint32_t seed) {
  uint32_t a = seed + threadIdx.x, b = seed * 3 + blockIdx.x;
  if (KIND == 0) {
    uint64_t acc[8];
#pragma unroll
    for (int j = 0; j < 8; j++) acc[j] = a + j;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 8; u++) {
#pragma unroll
        for (int j = 0; j < 8; j++)
          asm volatile("mad.wide.u32 %0, %1, %2, %0;" : "+l"(acc[j]) : "r"(a + u), "r"(b));
      }
    }
    uint64_t s = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) s ^= acc[j];
    if (s == 0x1234567) out[0] = (uint32_t)s;
  } else if (KIND == 1) {
    uint32_t acc[8];
#pragma unroll
    for (int j = 0; j < 8; j++) acc[j] = a + j;
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 8; u++) {
#pragma unroll
        for (int j = 0; j < 8; j++) asm volatile("mad.lo.u32 %0, %1, %2, %0;" : "+r"(acc[j]) : "r"(a + u), "r"(b));
      }
    }
    uint32_t s = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) s ^= acc[j];
    if (s == 0x1234567) out[0] = s;
  } else if (KIND == 3) {
    // carry OUT only: independent 64-bit accumulators, the carry of every product counted by an ALU-pipe addc
    uint64_t acc[8];
    uint32_t cnt[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      acc[j] = a + j;
      cnt[j] = 0;
    }
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 8; u++) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
          limb::mw_cc(acc[j], a + u, b + j, acc[j]);
          limb::addc(cnt[j], cnt[j], 0);
        }
      }
    }
    uint64_t s = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) s ^= acc[j] + cnt[j];
    if (s == 0x1234567) out[0] = (uint32_t)s;
  } else if (KIND == 4) {
    // carry IN only: an ALU-pipe add.cc produces the carry each IMAD.WIDE.X consumes; no carry out
    uint64_t acc[8];
    uint32_t src[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      acc[j] = a + j;
      src[j] = b + j;
    }
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 8; u++) {
#pragma unroll
        for (int j = 0; j < 8; j++) {
          limb::add_cc(src[j], src[j], a);
          limb::mwc(acc[j], a + u, b + j, acc[j]);
        }
      }
    }
    uint64_t s = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) s ^= acc[j] + src[j];
    if (s == 0x1234567) out[0] = (uint32_t)s;
  } else {
    // carry-chained pairs exactly as mont_row issues them: 2 independent chains of 8 limbs
    uint32_t x[8], y[8];
#pragma unroll
    for (int j = 0; j < 8; j++) {
      x[j] = a + j;
      y[j] = b + j;
    }
    for (int it = 0; it < iters; it++) {
#pragma unroll
      for (int u = 0; u < 8; u++) {
        limb::mad_lo_cc(x[0], a + u, b, x[0]);
        limb::madc_hi_cc(x[1], a + u, b, x[1]);
        limb::madc_lo_cc(x[2], a + u, y[2], x[2]);
        limb::madc_hi_cc(x[3], a + u, y[2], x[3]);
        limb::madc_lo_cc(x[4], a + u, y[4], x[4]);
        limb::madc_hi_cc(x[5], a + u, y[4], x[5]);
        limb::madc_lo_cc(x[6], a + u, y[6], x[6]);
        limb::madc_hi(x[7], a + u, y[6], x[7]);
        limb::mad_lo_cc(y[0], b + u, a, y[0]);
        limb::madc_hi_cc(y[1], b + u, a, y[1]);
        limb::madc_lo_cc(y[2], b + u, x[2], y[2]);
        limb::madc_hi_cc(y[3], b + u, x[2], y[3]);
        limb::madc_lo_cc(y[4], b + u, x[4], y[4]);
        limb::madc_hi_cc(y[5], b + u, x[4], y[5]);
        limb::madc_lo_cc(y[6], b + u, x[6], y[6]);
        limb::madc_hi(y[7], b + u, x[6], y[7]);
      }
    }
    uint32_t s = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) s ^= x[j] ^ y[j];
    if (s == 0x1234567) out[0] = s;
  }
}

extern "C" int ripp_bench_imad(ripp_ctx* ctx, int kind, int iters, double* macs_per_s, double* ms_out) {
  if (!ctx || !macs_per_s) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, ctx->device));
  void* out;
  OK(scratch(ctx, 3, 256, &out));
  int blocks = prop.multiProcessorCount * 8, threads = 256;
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  float best = 1e30f;
  for (int rep = 0; rep < 5; rep++) {
    CU(cudaEventRecord(e0, ctx->stream));
    if (kind == 0)
      k_imad<0><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, 12345u + rep);
    else if (kind == 1)
      k_imad<1><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, 12345u + rep);
    else if (kind == 3)
      k_imad<3><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, 12345u + rep);
    else if (kind == 4)
      k_imad<4><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, 12345u + rep);
    else
      k_imad<2><<<blocks, threads, 0, ctx->stream>>>((uint32_t*)out, iters, 12345u + rep);
    LAUNCHED(ctx);
    CU(cudaEventRecord(e1, ctx->stream));
    CU(cudaEventSynchronize(e1));
    float ms;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    if (rep > 0 && ms < best) best = ms;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  // MACs per thread per iteration: kind 0/1: 64; kind 2: 8 pairs x 2 chains x 8 = 64 pairs = 64 32x32 products
  double macs = (double)blocks * threads * (double)iters * 64.0;
  *macs_per_s = macs / (best * 1e-3);
  if (ms_out) *ms_out = best;
  return RIPP_OK;
}

// ------------------------------------------------------------------------------------------------
// L1: pairing inner product (the lane engines of pairing6.cu)
// ------------------------------------------------------------------------------------------------
extern "C" int ripp_pairing_ip_batch_dev(ripp_ctx* ctx, int nseg, const void* const* g1_aff_dev, const void* const* g2_aff_dev,
                                         size_t n, void* gt_out_dev) {
  if (!ctx || !g1_aff_dev || !g2_aff_dev || !gt_out_dev) return fail(RIPP_ERR_ARG, "null argument");
  return ripp_pairing_batch_l6(ctx, nseg, g1_aff_dev, g2_aff_dev, n, gt_out_dev, true);
}

extern "C" int ripp_miller_partial_dev(ripp_ctx* ctx, const void* g1, const void* g2, size_t n, void* out) {
  if (!ctx || !out || (n && (!g1 || !g2))) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  const void* a1[1] = {g1};
  const void* a2[1] = {g2};
  return ripp_pairing_batch_l6(ctx, 1, a1, a2, n, out, false);
}

extern "C" int ripp_gt_combine_dev(ripp_ctx* ctx, const void* partials, size_t count, void* out) {
  if (!ctx || !out || !partials || count == 0) return fail(RIPP_ERR_ARG, "bad argument");
  return ripp_final_exp_l6(ctx, partials, (uint32_t)count, out, 1);
}

// ---- batch primitives of the sharded (multi-GPU) provers: DESIGN.md §5 ---------------------------------------
// nseg Miller partials (no final exponentiation) of equal-length vector pairs in one launch
extern "C" int ripp_miller_partial_batch_dev(ripp_ctx* ctx, int nseg, const void* const* g1_aff_dev,
                                             const void* const* g2_aff_dev, size_t n, void* fq12_out_dev) {
  if (!ctx || !fq12_out_dev || !g1_aff_dev || !g2_aff_dev) return fail(RIPP_ERR_ARG, "null argument");
  return ripp_pairing_batch_l6(ctx, nseg, g1_aff_dev, g2_aff_dev, n, fq12_out_dev, false);
}
// out[s] = final_exponentiation(prod_r partials[s * count + r]), s < nseg
extern "C" int ripp_gt_combine_batch_dev(ripp_ctx* ctx, const void* partials, size_t count, int nseg, void* out) {
  if (!ctx || !out || !partials || count == 0 || nseg <= 0) return fail(RIPP_ERR_ARG, "bad argument");
  return ripp_final_exp_l6(ctx, partials, (uint32_t)count, out, nseg);
}
// out[s] = sum_r in[s * count + r] (G1 / G2 affine points or Fr), one thread per segment
template <class F>
__global__ void k_aff_seg_sum(const Aff<F>* __restrict__ in, uint32_t count, int nseg, Aff<F>* __restrict__ out) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  Jac<F> acc = Jac<F>::inf();
  for (uint32_t r = 0; r < count; r++) acc = acc.add_mixed(in[(size_t)s * count + r]);
  out[s] = acc.is_inf() ? Aff<F>::inf() : acc.to_affine();
}
__global__ void k_fr_seg_sum(const Fr* __restrict__ in, uint32_t count, int nseg, Fr* __restrict__ out) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= nseg) return;
  Fr acc = Fr::zero();
  for (uint32_t r = 0; r < count; r++) acc = acc + in[(size_t)s * count + r];
  out[s] = acc;
}
extern "C" int ripp_seg_sum_dev(ripp_ctx* ctx, int type, const void* in, size_t count, int nseg, void* out) {
  if (!ctx || !in || !out || count == 0 || nseg <= 0) return fail(RIPP_ERR_ARG, "bad argument");
  CU(cudaSetDevice(ctx->device));
  unsigned blk = (unsigned)((nseg + 31) / 32);
  if (type == 1)
    k_aff_seg_sum<Fq><<<blk, 32, 0, ctx->stream>>>((const G1Aff*)in, (uint32_t)count, nseg, (G1Aff*)out);
  else if (type == 2)
    k_aff_seg_sum<Fq2><<<blk, 32, 0, ctx->stream>>>((const G2Aff*)in, (uint32_t)count, nseg, (G2Aff*)out);
  else if (type == 3)
    k_fr_seg_sum<<<blk, 32, 0, ctx->stream>>>((const Fr*)in, (uint32_t)count, nseg, (Fr*)out);
  else
    return fail(RIPP_ERR_ARG, "type must be 1 (G1), 2 (G2) or 3 (Fr)");
  LAUNCHED(ctx);
  return RIPP_OK;
}

extern "C" int ripp_pairing_ip_dev(ripp_ctx* ctx, const void* g1, const void* g2, size_t n, void* out) {
  if (!ctx || !out || (n && (!g1 || !g2))) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  const void* a1[1] = {g1};
  const void* a2[1] = {g2};
  return ripp_pairing_batch_l6(ctx, 1, a1, a2, n, out, true);
}

static int pairing_ip_host(ripp_ctx* ctx, const void* g1, size_t nl, const void* g2, size_t nr, void* gt_out, bool jac) {
  if (!ctx || !gt_out) return fail(RIPP_ERR_ARG, "null argument");
  if (nl != nr)
    return fail(RIPP_ERR_LEN_MISMATCH,
                "left length, right length: " + std::to_string(nl) + ", " + std::to_string(nr));
  size_t n = nl;
  if (n && (!g1 || !g2)) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  void* dbuf;
  size_t s1 = jac ? sizeof(G1Jac) : sizeof(G1Aff), s2 = jac ? sizeof(G2Jac) : sizeof(G2Aff);
  size_t off_g2 = (n * s1 + 255) & ~(size_t)255;
  size_t off_a1 = off_g2 + ((n * s2 + 255) & ~(size_t)255);
  size_t off_a2 = off_a1 + ((n * sizeof(G1Aff) + 255) & ~(size_t)255);
  size_t off_out = off_a2 + ((n * sizeof(G2Aff) + 255) & ~(size_t)255);
  OK(scratch(ctx, 0, off_out + 1024, &dbuf));
  char* d = (char*)dbuf;
  const G1Aff* pa;
  const G2Aff* qa;
  if (n) {
    CU(cudaMemcpyAsync(d, g1, n * s1, cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d + off_g2, g2, n * s2, cudaMemcpyHostToDevice, ctx->stream));
  }
  if (jac && n) {
    k_normalize<Fq><<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>((const G1Jac*)d, (G1Aff*)(d + off_a1), n);
    LAUNCHED(ctx);
    k_normalize<Fq2><<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>((const G2Jac*)(d + off_g2), (G2Aff*)(d + off_a2), n);
    LAUNCHED(ctx);
    pa = (const G1Aff*)(d + off_a1);
    qa = (const G2Aff*)(d + off_a2);
  } else {
    pa = (const G1Aff*)d;
    qa = (const G2Aff*)(d + off_g2);
  }
  OK(ripp_pairing_ip_dev(ctx, pa, qa, n, d + off_out));
  CU(cudaMemcpyAsync(gt_out, d + off_out, sizeof(Fq12), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}

extern "C" int ripp_pairing_ip(ripp_ctx* ctx, const void* g1_jac, size_t nl, const void* g2_jac, size_t nr, void* gt_out) {
  return pairing_ip_host(ctx, g1_jac, nl, g2_jac, nr, gt_out, true);
}
extern "C" int ripp_pairing_ip_affine(ripp_ctx* ctx, const void* g1, size_t nl, const void* g2, size_t nr, void* gt_out) {
  return pairing_ip_host(ctx, g1, nl, g2, nr, gt_out, false);
}
