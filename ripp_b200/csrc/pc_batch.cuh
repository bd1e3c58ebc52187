// Commit to and open `count` polynomials under one key in one call (include/ripp_b200.h "ripp_pc_commit_batch_dev",
// "ripp_pc_open_batch_dev").  Part of the gipa.cu translation unit, after poly_commit.cuh and aggregate_batch.cuh, whose
// serialisation, Fiat-Shamir helpers, segment tables and staging it shares; result k is byte for byte what the single
// entry point returns for instance k alone.
//
// Every vector lives in one arena per vector, instance k at element k n (second tier) or k m (first tier).  Then:
//   commit     one table-driven gather of the zero-padded coefficients, ONE segmented MSM of count n rows over the
//              shared first-tier bases, ONE pairing chain for the count AFGHO products, one copy, one sync;
//   open       the powers of every x_k (and y_k), the row combinations, y_eval_comm as one segmented MSM; trusted: the
//              division of every y_eval_k by (X - y_k) as one segmented scan and the count KZG proofs as one MSM;
//              transparent: the count evaluations as one segmented dot product;
//   rounds     the count second-tier recursions (MULTIEXP_SSM) and, transparent, the count first-tier recursions
//              (SCALAR_SSM_G1) in lock step, both tiers sharing a round: one pairing chain for the 2 count products,
//              two segmented G1 MSMs per tier, one segmented Fr dot product launch, one copy, one sync, host challenges,
//              one fold-table launch per tier;
//   closing    the base values gathered and copied once; trusted: the final keys' KZG quotients on host threads and
//              one segmented G2 MSM over h_beta_powers.
// The number of launches and synchronisations depends on (kind, n, m), not on count.
#pragma once

// one polynomial of the batch: its coefficients and their number (layout of "Coefficient layout")
struct PcPoly {
  const Fr* c;
  size_t len;
};

// out[k nm + e] = C_k[e], zero from len_k on
__global__ void k_pc_gather(const PcPoly* __restrict__ polys, size_t nm, size_t count, Fr* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count * nm) return;
  size_t k, e;
  pc::seg_split(i, nm, &k, &e);
  const PcPoly p = polys[k];
  out[i] = e < p.len ? p.c[e] : Fr::zero();
}

// out[k n + e] = base[k]^e (base 0 gives 1, 0, 0, ...)
__global__ void k_pc_powers_seg(const Fr* __restrict__ base, size_t n, size_t total, Fr* __restrict__ out) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  size_t k, e;
  pc::seg_split(i, n, &k, &e);
  out[i] = pc::pow(base[k], e);
}

// k_pc_rows per instance: part[(k G + g) m + j] = sum_{i in [g R, (g+1) R), i < n} x_k^(i - g R) C_k[i m + j]
__global__ void k_pc_rows_seg(const PcPoly* __restrict__ polys, const Fr* __restrict__ x, size_t m, size_t n, size_t G, size_t R,
                              size_t count, Fr* __restrict__ part) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count * G * m) return;
  size_t k, g, j;
  pc::row_index(t, G, m, &k, &g, &j);
  const PcPoly p = polys[k];
  const Fr xk = x[k];
  const size_t lo = g * R, hi = lo + R < n ? lo + R : n;
  Fr acc = Fr::zero();
  for (size_t i = hi; i-- > lo;) {
    const size_t at = i * m + j;
    acc = pc::horner_step(acc, xk, at < p.len ? p.c[at] : Fr::zero());
  }
  part[t] = acc;
}

// k_pc_rows_combine per instance: y[k m + j] = sum_g x_k^(g R) part[(k G + g) m + j]
__global__ void k_pc_rows_combine_seg(const Fr* __restrict__ part, const Fr* __restrict__ x, size_t m, size_t G, size_t R, size_t count,
                                      Fr* __restrict__ y) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count * m) return;
  size_t k, j;
  pc::seg_split(t, m, &k, &j);
  const Fr xr = pc::pow(x[k], R);
  const Fr* pk = part + k * G * m + j;
  Fr acc = Fr::zero();
  for (size_t g = G; g-- > 0;) acc = pc::horner_step(acc, xr, pk[g * m]);
  y[t] = acc;
}

// k_pc_div_heads over count segments of N at scan level `level` (point z_k^(L^level)): heads[k nb + b]
__global__ void k_pc_div_heads_seg(const Fr* __restrict__ c, size_t N, size_t count, const Fr* __restrict__ z, unsigned level,
                                   Fr* __restrict__ heads) {
  const size_t nb = (N + PC_CHUNK - 1) / PC_CHUNK;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count * nb) return;
  size_t k, b;
  pc::seg_split(t, nb, &k, &b);
  const size_t lo = b * PC_CHUNK, hi = lo + PC_CHUNK < N ? lo + PC_CHUNK : N;
  heads[t] = pc::chunk_head(c + k * N, lo, hi, pc::pow2k(z[k], 5 * level), Fr::zero());
}

// k_pc_div_replay over count segments: S the carries (k nb + b; NULL when nb == 1); segment k writes s_0 to
// out0[k s0] and s_e to out[k so + e - 1]
__global__ void k_pc_div_replay_seg(const Fr* __restrict__ c, size_t N, size_t count, const Fr* __restrict__ z, unsigned level,
                                    const Fr* __restrict__ S, Fr* out0, size_t s0, Fr* out, size_t so) {
  const size_t nb = (N + PC_CHUNK - 1) / PC_CHUNK;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count * nb) return;
  size_t k, b;
  pc::seg_split(t, nb, &k, &b);
  const size_t lo = b * PC_CHUNK, hi = lo + PC_CHUNK < N ? lo + PC_CHUNK : N;
  pc::chunk_replay(c + k * N, lo, hi, pc::pow2k(z[k], 5 * level), hi < N ? S[t + 1] : Fr::zero(), out0 + k * s0, out + k * so);
}

// where the two halves of a segmented dot product read: segment s = p K + k of instance k at a + k stride + a_off[p]
struct PcDot {
  size_t a_off[2], b_off[2];
};

// out[s nch + ch] = sum over chunk ch (R elements) of a_s[e] b_s[e] (b NULL: a_s[e]), e < h
__global__ void k_pc_dot_seg(const Fr* __restrict__ a, const Fr* __restrict__ b, size_t stride, size_t K, size_t nseg, size_t h,
                             uint32_t R, PcDot o, Fr* __restrict__ out) {
  const size_t nch = (h + R - 1) / R;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= nseg * nch) return;
  size_t s, ch, p, k;
  pc::seg_split(t, nch, &s, &ch);
  pc::seg_split(s, K, &p, &k);
  const Fr* as = a + k * stride + (p ? o.a_off[1] : o.a_off[0]);  // selects, not an indexed (local memory) read
  const Fr* bs = b ? b + k * stride + (p ? o.b_off[1] : o.b_off[0]) : nullptr;
  const size_t lo = ch * R, hi = lo + R < h ? lo + R : h;
  Fr acc = Fr::zero();
  for (size_t e = lo; e < hi; e++) acc = acc + (bs ? as[e] * bs[e] : as[e]);
  out[t] = acc;
}

// Fr of workspace seg_dot needs for nseg dot products of length h
static size_t dot_tmp_len(size_t nseg, size_t h) {
  const size_t nch = (h + 15) / 16;
  return nch > 1 ? 2 * nseg * nch : 0;
}

// out[s] = <a_s, b_s> for nseg segments of length h >= 1 (PcDot layout): one launch per level of 16, log16 h levels
static int seg_dot(ripp_ctx* ctx, const Fr* a, const Fr* b, size_t stride, size_t K, size_t nseg, size_t h, const PcDot& o, Fr* tmp,
                   Fr* out) {
  const uint32_t R = 16;
  size_t nch = (h + R - 1) / R;
  Fr *pa = tmp, *pb = tmp + nseg * nch;
  k_pc_dot_seg<<<(unsigned)((nseg * nch + 127) / 128), 128, 0, ctx->stream>>>(a, b, stride, K, nseg, h, R, o, nch == 1 ? out : pa);
  LAUNCHED(ctx);
  const PcDot flat = {{0, 0}, {0, 0}};
  while (nch > 1) {
    const size_t no = (nch + R - 1) / R;
    k_pc_dot_seg<<<(unsigned)((nseg * no + 127) / 128), 128, 0, ctx->stream>>>(pa, nullptr, nch, nseg, nseg, nch, R, flat,
                                                                                no == 1 ? out : pb);
    LAUNCHED(ctx);
    Fr* t = pa;
    pa = pb;
    pb = t;
    nch = no;
  }
  return RIPP_OK;
}

// div_scan over count segments of N at level `level`: tmp count div_tmp_len(N) Fr
static int div_scan_seg(ripp_ctx* ctx, const Fr* c, size_t N, size_t count, const Fr* z, unsigned level, Fr* tmp, Fr* out0, size_t s0,
                        Fr* out, size_t so) {
  const size_t nb = (N + PC_CHUNK - 1) / PC_CHUNK;
  const unsigned blocks = (unsigned)((count * nb + 127) / 128);
  Fr* S = nullptr;
  if (nb > 1) {
    Fr* heads = tmp;
    S = tmp + count * nb;
    k_pc_div_heads_seg<<<blocks, 128, 0, ctx->stream>>>(c, N, count, z, level, heads);
    LAUNCHED(ctx);
    OK(div_scan_seg(ctx, heads, nb, count, z, level + 1, tmp + 2 * count * nb, S, nb, S + 1, nb));
  }
  k_pc_div_replay_seg<<<blocks, 128, 0, ctx->stream>>>(c, N, count, z, level, S, out0, s0, out, so);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// the single path's checks in its order, its limits over the whole batch (count n rows, count n m coefficients)
static int pc_batch_check(bool trusted_open, size_t m, size_t n, size_t count, const void* const* coeffs, const size_t* lens) {
  for (size_t k = 0; k < count; k++)
    if (lens[k] && !coeffs[k]) return fail(RIPP_ERR_ARG, "null argument: coefficients of polynomial " + std::to_string(k));
  OK(pc_shape(n, m, 0));
  if (trusted_open && n < 2) return fail(RIPP_ERR_ARG, "the trusted opening needs at least two rows (TIPA of length 1)");
  for (size_t k = 0; k < count; k++)
    if (lens[k] > n * m) return fail(RIPP_ERR_ARG, "polynomial " + std::to_string(k) + ": len > rows x row length");
  if (count > ((size_t)1 << 16) / n || count * n > ((size_t)1 << 24) / m)
    return fail(RIPP_ERR_ARG, "polynomial commitment batch: more than 2^16 rows or 2^24 coefficients in all");
  return RIPP_OK;
}

static int upload_polys(ripp_ctx* ctx, size_t count, const void* const* coeffs, const size_t* lens, PcPoly* dev) {
  std::vector<PcPoly> t(count);
  for (size_t k = 0; k < count; k++) t[k] = PcPoly{(const Fr*)coeffs[k], lens[k]};
  uint8_t* pin;
  OK(pinned_grow(ctx, count * sizeof(PcPoly), &pin));
  memcpy(pin, t.data(), count * sizeof(PcPoly));
  CU(cudaMemcpyAsync(dev, pin, count * sizeof(PcPoly), cudaMemcpyHostToDevice, ctx->stream));
  return RIPP_OK;
}

extern "C" int ripp_pc_commit_batch_dev(ripp_ctx* ctx, const void* first_tier_dev, size_t m, const void* second_tier_dev, size_t n,
                                        size_t count, const void* const* coeffs_dev, const size_t* lens, void* gt_out,
                                        void* y_coms_dev) {
  if (!ctx || !first_tier_dev || !second_tier_dev || (count && (!coeffs_dev || !lens || !gt_out || !y_coms_dev)))
    return fail(RIPP_ERR_ARG, "null argument");
  OK(pc_batch_check(false, m, n, count, coeffs_dev, lens));
  if (count == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const size_t K = count, rows = K * n, N = rows * m;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  // workspace: polynomial table | segment table | GT results | padded coefficients
  const size_t o_tab = 0, o_segs = o_tab + up(K * sizeof(PcPoly)), o_gt = o_segs + up(K * sizeof(M6SegH)), o_c = o_gt + up(K * 576),
               ws_bytes = o_c + N * sizeof(Fr);
  void* ws;
  OK(scratch(ctx, 48, ws_bytes, &ws));
  char* W = (char*)ws;
  PcPoly* tab = (PcPoly*)(W + o_tab);
  OK(upload_polys(ctx, K, coeffs_dev, lens, tab));
  {
    std::vector<M6SegH> segs(K);
    for (size_t k = 0; k < K; k++) segs[k] = M6SegH{(const char*)y_coms_dev + k * n * 96, second_tier_dev};
    CU(cudaMemcpyAsync(W + o_segs, segs.data(), K * sizeof(M6SegH), cudaMemcpyHostToDevice, st));
  }
  k_pc_gather<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(tab, n * m, K, (Fr*)(W + o_c));
  LAUNCHED(ctx);
  OK(ripp_msm_batch_internal(ctx, 1, first_tier_dev, 0, W + o_c, m, m, rows, y_coms_dev));
  OK(ripp_pairing_table_l6(ctx, W + o_segs, K, n, W + o_gt, 44));
  CU(cudaMemcpyAsync(gt_out, W + o_gt, K * 576, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return RIPP_OK;
}

// bytes of one batched OpeningProof: trusted TIPAWithSSM (GIPA rounds, r_base, ck_base, KZG opening) || y_eval_comm ||
// kzg_proof; transparent second-tier GIPA || y_eval_comm || first-tier GIPA
static size_t pc_proof_len(int kind, size_t L2, size_t L1) {
  const size_t second = 8 + L2 * 2 * (576 + 32 + 8 + 96) + 96 + 32;
  if (kind == RIPP_PC_TRUSTED) return second + 192 + 192 + 96 + 96;
  return second + 96 + 8 + L1 * 2 * (96 + 32 + 8 + 32) + 32 + 32;
}

static int pc_open_batch(ripp_ctx* ctx, int kind, const void* first_tier, size_t m, const void* second_tier, size_t n,
                         const void* srs_g2, size_t K, const void* const* coeffs, const size_t* lens, const void* y_coms,
                         const Fr* xs, const Fr* ys, uint8_t* proofs_out, size_t len, void* evals_out) {
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  const bool trusted = kind == RIPP_PC_TRUSTED;
  size_t L2 = 0, L1 = 0;
  while (((size_t)1 << L2) < n) L2++;
  while (((size_t)1 << L1) < m) L1++;
  if (trusted) L1 = 0;  // the first tier is a KZG opening, not a recursion
  const size_t Nn = K * n, Nm = K * m;
  size_t G, R;
  pc::row_groups_batch(K, n, m, &G, &R);
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  // ---- arenas: powers of x / B2 (K n Fr), A2 (K n G1), V2 (K n G2), y_eval / A1 (K m Fr), quotient or powers of y / B1
  // (K m Fr), V1 (K m G1, transparent), row partials, scan or dot workspace ----
  const size_t tmp_fr = trusted ? K * div_tmp_len(m) : dot_tmp_len(2 * K, m / 2 > 0 ? m / 2 : 1) + dot_tmp_len(K, m);
  const size_t o_B2 = 0, o_A2 = o_B2 + up(Nn * 32), o_V2 = o_A2 + up(Nn * 96), o_A1 = o_V2 + up(Nn * 192), o_B1 = o_A1 + up(Nm * 32),
               o_V1 = o_B1 + up(Nm * 32), o_part = o_V1 + (trusted ? 0 : up(Nm * 96)), o_tmp = o_part + (G > 1 ? up(K * G * m * 32) : 0),
               ar_bytes = o_tmp + up(tmp_fr * 32 + 32);
  void* ar;
  OK(scratch(ctx, 49, ar_bytes, &ar));
  char* AR = (char*)ar;
  Fr *B2 = (Fr*)(AR + o_B2), *A1 = (Fr*)(AR + o_A1), *B1 = (Fr*)(AR + o_B1), *tmp = (Fr*)(AR + o_tmp);
  char *A2 = AR + o_A2, *V2 = AR + o_V2, *V1 = AR + o_V1;
  // ---- workspace: polynomial table, points, segment tables, round results, fold records, base values ----
  const size_t nseg_all = 2 * K * L2;
  const size_t rec_bytes = 3 * K * sizeof(EndoBits) + 3 * K * 32;
  const size_t res_bytes = 2 * K * (576 + 96 + 96 + 32);
  const size_t base_bytes = K * (96 + 32 + 192 + 32 + 32 + 96 + 96 + 32);  // A2 B2 V2 A1 B1 base values, y_eval_comm, kzg, evals
  const size_t o_tab = 0, o_xy = o_tab + up(K * sizeof(PcPoly)), o_segs = o_xy + up(2 * K * 32),
               o_res = o_segs + up(nseg_all * sizeof(M6SegH)), o_rec = o_res + up(res_bytes), o_pts = o_rec + up(rec_bytes),
               o_ev = o_pts + up(2 * K * 96), o_base = o_ev + up(K * 32), ws_bytes = o_base + up(base_bytes);
  void* ws;
  OK(scratch(ctx, 50, ws_bytes, &ws));
  char* WS = (char*)ws;
  PcPoly* tab = (PcPoly*)(WS + o_tab);
  Fr* xy = (Fr*)(WS + o_xy);
  G1Aff* pts = (G1Aff*)(WS + o_pts);  // y_eval_comm (K), kzg proofs (K)
  Fr* ev = (Fr*)(WS + o_ev);
  char* res = WS + o_res;
  // page-locked staging: results at the front, the fold records behind them
  const size_t pin_res = res_bytes > base_bytes ? res_bytes : base_bytes;
  const size_t pin_bytes = up(pin_res) + up(rec_bytes > 2 * K * 32 ? rec_bytes : 2 * K * 32) + up(K * sizeof(PcPoly));
  uint8_t* pin;
  OK(pinned_grow(ctx, pin_bytes, &pin));
  uint8_t* pup = pin + up(pin_res);
  ripp_ctx* mk2 = ripp_child(ctx, 0);
  ripp_ctx* mk1 = ripp_child(ctx, 1);
  if (!mk2 || !mk1) return fail(RIPP_ERR_CUDA, "child context");

  // ---- tables, points, second-tier vectors ----
  {
    PcPoly* t = (PcPoly*)(pup + up(rec_bytes > 2 * K * 32 ? rec_bytes : 2 * K * 32));
    for (size_t k = 0; k < K; k++) t[k] = PcPoly{(const Fr*)coeffs[k], lens[k]};
    CU(cudaMemcpyAsync(tab, t, K * sizeof(PcPoly), cudaMemcpyHostToDevice, st));
    memcpy(pup, xs, K * 32);
    memcpy(pup + K * 32, ys, K * 32);
    CU(cudaMemcpyAsync(xy, pup, 2 * K * 32, cudaMemcpyHostToDevice, st));
    std::vector<M6SegH> segs(nseg_all);
    size_t s = 0;
    for (size_t h = n / 2; h >= 1; h /= 2)  // gipa.rs:209-231 -- IP(A_R, v_L), IP(A_L, v_R) of every instance
      for (int p = 0; p < 2; p++)
        for (size_t k = 0; k < K; k++)
          segs[s++] = p == 0 ? M6SegH{A2 + (k * n + h) * 96, V2 + k * n * 192} : M6SegH{A2 + k * n * 96, V2 + (k * n + h) * 192};
    if (nseg_all) CU(cudaMemcpyAsync(WS + o_segs, segs.data(), nseg_all * sizeof(M6SegH), cudaMemcpyHostToDevice, st));
  }
  const M6SegH* segs_dev = (const M6SegH*)(WS + o_segs);
  const Fr *xd = xy, *yd = xy + K;
  CU(cudaMemcpyAsync(A2, y_coms, Nn * 96, cudaMemcpyDeviceToDevice, st));
  k_gather_rows<<<(unsigned)((Nn * 48 + 127) / 128), 128, 0, st>>>((const uint32_t*)second_tier, 0, (uint32_t)(n * 48), K, (uint32_t*)V2);
  LAUNCHED(ctx);
  k_pc_powers_seg<<<(unsigned)((Nn + 127) / 128), 128, 0, st>>>(xd, n, Nn, B2);
  LAUNCHED(ctx);
  // ---- mod.rs:221-241 / transparent.rs after :137: y_eval, y_eval_comm ----
  Fr* part = G > 1 ? (Fr*)(AR + o_part) : A1;
  k_pc_rows_seg<<<(unsigned)pc::row_blocks(K, G, m), 128, 0, st>>>(tab, xd, m, n, G, R, K, part);
  LAUNCHED(ctx);
  if (G > 1) {
    k_pc_rows_combine_seg<<<(unsigned)((Nm + 127) / 128), 128, 0, st>>>(part, xd, m, G, R, K, A1);
    LAUNCHED(ctx);
  }
  OK(ripp_msm_batch_internal(ctx, 1, first_tier, 0, A1, m, m, K, pts));
  if (trusted) {
    // KZG::open(kzg, y_eval_k, y_k) (mod.rs:98-104): quotients at stride m, y_eval_k(y_k) = f_k(x_k, y_k)
    OK(div_scan_seg(ctx, A1, m, K, yd, 0, tmp, ev, 1, B1, m));
    OK(ripp_msm_batch_internal(ctx, 1, first_tier, 0, B1, m, m - 1, K, pts + K));
  } else {
    // powers of y_k, f_k(x_k, y_k) = <y_eval_k, powers of y_k>, the replicated first-tier key
    k_pc_powers_seg<<<(unsigned)((Nm + 127) / 128), 128, 0, st>>>(yd, m, Nm, B1);
    LAUNCHED(ctx);
    const PcDot flat = {{0, 0}, {0, 0}};
    OK(seg_dot(ctx, A1, B1, m, K, K, m, flat, tmp, ev));
    k_gather_rows<<<(unsigned)((Nm * 24 + 127) / 128), 128, 0, st>>>((const uint32_t*)first_tier, 0, (uint32_t)(m * 24), K, (uint32_t*)V1);
    LAUNCHED(ctx);
  }

  // ---- rounds in lock step: the second tier over n, the transparent first tier over m ----
  std::vector<std::vector<Bytes>> steps2(K), steps1(K);  // per instance: serialised rounds, oldest first
  std::vector<std::vector<Fr>> tr2(K), tr1(K);
  const Fr zero = Fr::zero();
  // Fr [c2^-1][c1][c1^-1] first (Fr is 16-byte aligned, an EndoBits 168 bytes long), then [G1 c2][G2 c2^-1][G1 c1^-1]
  Fr* rec_fr = (Fr*)pup;
  EndoBits* rec = (EndoBits*)(rec_fr + 3 * K);
  const Fr* rdf = (const Fr*)(WS + o_rec);
  const EndoBits* rd = (const EndoBits*)(rdf + 3 * K);
  char *r2gt = res, *r2g1 = res + 2 * K * 576, *r1g1 = r2g1 + 2 * K * 96, *r1fr = r1g1 + 2 * K * 96;
  const size_t rounds = L2 > L1 ? L2 : L1;
  for (size_t round = 0; round < rounds; round++) {
    const size_t h2 = round < L2 ? n >> (round + 1) : 0, h1 = round < L1 ? m >> (round + 1) : 0;
    double t_r0 = now_ms();
    if (h2) {  // gipa.rs:209-231 -- IP(A_R, B_L), IP(A_L, B_R) as two segmented MSMs, IP(A_R, v_L), IP(A_L, v_R) as one chain
      OK(ripp_fork(ctx, mk2));
      OK(ripp_msm_batch_internal(mk2, 1, A2 + h2 * 96, n, B2, n, h2, K, r2g1));
      OK(ripp_msm_batch_internal(mk2, 1, A2, n, B2 + h2, n, h2, K, r2g1 + K * 96));
    }
    if (h1) {  // IP(A_R, v_L), IP(A_L, v_R) over the per-instance keys; IP(A_R, B_L), IP(A_L, B_R) as one dot launch
      OK(ripp_fork(ctx, mk1));
      OK(ripp_msm_batch_internal(mk1, 1, V1, m, A1 + h1, m, h1, K, r1g1));
      OK(ripp_msm_batch_internal(mk1, 1, V1 + h1 * 96, m, A1, m, h1, K, r1g1 + K * 96));
      const PcDot halves = {{h1, 0}, {0, h1}};
      OK(seg_dot(ctx, A1, B1, m, K, 2 * K, h1, halves, tmp, (Fr*)r1fr));
    }
    if (h2) OK(ripp_pairing_table_l6(ctx, segs_dev + round * 2 * K, 2 * K, h2, r2gt, 44));
    if (h2) OK(ripp_join(ctx, mk2));
    if (h1) OK(ripp_join(ctx, mk1));
    CU(cudaMemcpyAsync(pin, res, res_bytes, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    // gipa.rs:235-258 -- Fiat-Shamir challenges and the fold scalars' records
    host_parallel((h2 ? K : 0) + (h1 ? K : 0), 64, [&](size_t i) {
      Val v[6];
      Fr c, ci;
      const bool second = h2 && i < K;  // the second tier's K items first
      const size_t k = i % K;
      const uint8_t* P = pin;
      if (second) {
        v[0] = val_of(VT_GT, P + k * 576);
        v[2] = val_of(VT_G1, P + 2 * K * 576 + k * 96);
        v[3] = val_of(VT_GT, P + (K + k) * 576);
        v[5] = val_of(VT_G1, P + 2 * K * 576 + (K + k) * 96);
      } else {
        const uint8_t* g1 = P + 2 * K * 576 + 2 * K * 96;
        const uint8_t* fr = g1 + 2 * K * 96;
        v[0] = val_of(VT_G1, g1 + k * 96);
        v[2] = val_of(VT_FR, fr + k * 32);
        v[3] = val_of(VT_G1, g1 + (K + k) * 96);
        v[5] = val_of(VT_FR, fr + (K + k) * 32);
      }
      v[1] = val_of(VT_FR, nullptr);  // SSMPlaceholderCommitment
      v[4] = val_of(VT_FR, nullptr);
      std::vector<Fr>& tr = second ? tr2[k] : tr1[k];
      gipa_challenge(tr.empty() ? zero : tr.back(), v, &c, &ci);
      tr.push_back(c);
      if (second) {
        ripp_endo_bits(1, c.v, &rec[k]);
        ripp_endo_bits(2, ci.v, &rec[K + k]);
        rec_fr[k] = ci;
      } else {
        ripp_endo_bits(1, ci.v, &rec[2 * K + k]);
        rec_fr[K + k] = c;
        rec_fr[2 * K + k] = ci;
      }
      Bytes chunk;
      for (int j = 0; j < 6; j++) {
        if (j % 3 == 2) put_u64_le(chunk, 1);
        put_val(chunk, v[j]);
      }
      (second ? steps2[k] : steps1[k]).push_back(std::move(chunk));
    });
    // gipa.rs:261-291 -- A <- A_R c + A_L, B <- B_R c^-1 + B_L, v <- v_R c^-1 + v_L: one table per tier
    CU(cudaMemcpyAsync(WS + o_rec, pup, rec_bytes, cudaMemcpyHostToDevice, st));
    if (h2) {
      FoldTable ft;
      memset(&ft, 0, sizeof(ft));
      ft.K = (uint32_t)K;
      ft.n = (uint32_t)h2;
      ft.ngroups[0] = 1, ft.base[0][0] = A2, ft.sc[0][0] = rd, ft.stride[0][0] = n * 96;
      ft.ngroups[1] = 1, ft.base[1][0] = V2, ft.sc[1][0] = rd + K, ft.stride[1][0] = n * 192;
      ft.ngroups[2] = 1, ft.base[2][0] = (char*)B2, ft.sc[2][0] = rdf, ft.stride[2][0] = n * 32;
      OK(ripp_fold_table_internal(ctx, ft));
    }
    if (h1) {
      FoldTable ft;
      memset(&ft, 0, sizeof(ft));
      ft.K = (uint32_t)K;
      ft.n = (uint32_t)h1;
      ft.ngroups[0] = 1, ft.base[0][0] = V1, ft.sc[0][0] = rd + 2 * K, ft.stride[0][0] = m * 96;
      ft.ngroups[2] = 2, ft.base[2][0] = (char*)A1, ft.sc[2][0] = rdf + K, ft.stride[2][0] = m * 32;
      ft.base[2][1] = (char*)B1, ft.sc[2][1] = rdf + 2 * K, ft.stride[2][1] = m * 32;
      OK(ripp_fold_table_internal(ctx, ft));
    }
    if (trace_on()) fprintf(stderr, "[trace] pc open batch round %zu (n' = %zu, m' = %zu) %.2f ms\n", round, h2, h1, now_ms() - t_r0);
  }

  // ---- base values, y_eval_comm, kzg proofs, evaluations: one copy, one sync ----
  struct Part {
    const char* src;
    size_t stride_words, esz;
  };
  const Part parts[8] = {{A2, n * 24, 96},       {(const char*)B2, n * 8, 32}, {V2, n * 48, 192},       {(const char*)A1, m * 8, 32},
                         {(const char*)B1, m * 8, 32}, {(const char*)pts, 24, 96}, {(const char*)(pts + K), 24, 96}, {(const char*)ev, 8, 32}};
  size_t off[9];
  off[0] = 0;
  char* base = WS + o_base;
  for (int i = 0; i < 8; i++) {
    const uint32_t words = (uint32_t)(parts[i].esz / 4);
    k_gather_rows<<<(unsigned)((K * words + 127) / 128), 128, 0, st>>>((const uint32_t*)parts[i].src, parts[i].stride_words, words, K,
                                                                      (uint32_t*)(base + off[i]));
    LAUNCHED(ctx);
    off[i + 1] = off[i] + K * parts[i].esz;
  }
  CU(cudaMemcpyAsync(pin, base, off[8], cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  auto at = [&](int i, size_t k) { return pin + off[i] + k * parts[i].esz; };
  std::vector<uint8_t> opens;
  if (trusted) {
    // tipa/mod.rs:195-209, structured_scalar_message.rs:238-251: the final keys' openings with shift 1
    const size_t n_srs = 2 * n - 1;
    double t_o0 = now_ms();
    void* qd;
    OK(scratch(ctx, 51, up(K * n_srs * sizeof(Fr)) + K * 192, &qd));
    std::vector<Fr> q(K * n_srs);
    host_parallel(K, n >= 256 ? 1 : 16, [&](size_t k) {
      std::vector<Fr> rev(tr2[k].rbegin(), tr2[k].rend()), tinv(rev.size());
      for (size_t j = 0; j < rev.size(); j++) tinv[j] = rev[j].inv();
      Bytes p;
      put_fr(p, rev[0]);
      put_val(p, val_of(VT_G2, at(2, k)));
      const Fr z = challenge_from_random_bytes(p);
      std::vector<Fr> qk = kzg_quotient(tinv, Fr::one(), z, n_srs);
      memcpy(&q[k * n_srs], qk.data(), n_srs * sizeof(Fr));
    });
    CU(cudaMemcpyAsync(qd, q.data(), q.size() * sizeof(Fr), cudaMemcpyHostToDevice, st));
    char* od = (char*)qd + up(K * n_srs * sizeof(Fr));
    OK(ripp_msm_batch_internal(ctx, 2, srs_g2, 0, qd, n_srs, n_srs, K, od));
    opens.resize(K * 192);
    CU(cudaMemcpyAsync(opens.data(), od, K * 192, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (trace_on()) fprintf(stderr, "[trace] pc open batch openings %.2f ms\n", now_ms() - t_o0);
  }

  // ---- OpeningProofs (mod.rs:145-149 / transparent.rs:79-83) ----
  std::vector<int> bad(K, 0);
  host_parallel(K, 16, [&](size_t k) {
    Bytes out;
    out.reserve(len);
    put_u64_le(out, L2);
    for (size_t i = L2; i-- > 0;) out.insert(out.end(), steps2[k][i].begin(), steps2[k][i].end());
    put_val(out, val_of(VT_G1, at(0, k)));
    put_val(out, val_of(VT_FR, at(1, k)));
    if (trusted) {
      put_val(out, val_of(VT_G2, at(2, k)));
      put_val(out, val_of(VT_G2, opens.data() + k * 192));
      put_val(out, val_of(VT_G1, at(5, k)));
      put_val(out, val_of(VT_G1, at(6, k)));
    } else {
      put_val(out, val_of(VT_G1, at(5, k)));
      put_u64_le(out, L1);
      for (size_t i = L1; i-- > 0;) out.insert(out.end(), steps1[k][i].begin(), steps1[k][i].end());
      put_val(out, val_of(VT_FR, at(3, k)));
      put_val(out, val_of(VT_FR, at(4, k)));
    }
    if (out.size() != len) {
      bad[k] = 1;
      return;
    }
    memcpy(proofs_out + k * len, out.data(), len);
  });
  for (size_t k = 0; k < K; k++)
    if (bad[k]) return fail(RIPP_ERR_CUDA, "polynomial " + std::to_string(k) + ": proof length differs from the layout");
  if (evals_out)
    for (size_t k = 0; k < K; k++) memcpy((uint8_t*)evals_out + k * 32, at(7, k), 32);
  return RIPP_OK;
}

extern "C" int ripp_pc_open_batch_dev(ripp_ctx* ctx, int kind, const void* first_tier_dev, size_t m, const void* second_tier_dev,
                                      size_t n, const void* srs_g2_dev, size_t count, const void* const* coeffs_dev, const size_t* lens,
                                      const void* y_coms_dev, const void* x_host, const void* y_host, uint8_t* proofs_out,
                                      size_t proofs_cap, size_t* proof_len, void* evals_out) {
  if (!ctx || !first_tier_dev || !second_tier_dev || !proof_len ||
      (count && (!coeffs_dev || !lens || !y_coms_dev || !x_host || !y_host)))
    return fail(RIPP_ERR_ARG, "null argument");
  if (kind != RIPP_PC_TRUSTED && kind != RIPP_PC_TRANSPARENT) return fail(RIPP_ERR_ARG, "bad polynomial-commitment kind");
  if (kind == RIPP_PC_TRUSTED && !srs_g2_dev) return fail(RIPP_ERR_ARG, "the trusted opening needs h_beta_powers");
  OK(pc_batch_check(kind == RIPP_PC_TRUSTED, m, n, count, coeffs_dev, lens));
  if (count == 0) {
    *proof_len = 0;
    return RIPP_OK;
  }
  size_t L2 = 0, L1 = 0;
  while (((size_t)1 << L2) < n) L2++;
  while (((size_t)1 << L1) < m) L1++;
  const size_t len = pc_proof_len(kind, L2, L1);
  *proof_len = len;
  if (!proofs_out || proofs_cap / len < count) return fail(RIPP_ERR_ARG, "output buffer too small: need " + std::to_string(count * len));
  return pc_open_batch(ctx, kind, first_tier_dev, m, second_tier_dev, n, srs_g2_dev, count, coeffs_dev, lens, y_coms_dev,
                       (const Fr*)x_host, (const Fr*)y_host, proofs_out, len, evals_out);
}
