// aggregate_proofs for `count` independent batches of n proofs under one SRS, in one call (include/ripp_b200.h
// "ripp_tipp_aggregate_batch_dev").  Part of the gipa.cu translation unit, whose serialisation and Fiat-Shamir helpers it
// shares; proof k is byte for byte what ripp_tipp_aggregate_dev returns for batch k alone.
//
// The single prover is a chain of latency-bound rounds: per GIPA round one Miller / reduce / final-exponentiation chain,
// one host synchronisation for the challenge, one fold launch.  Here the 2K recursions of K batches (K of kind PAIRING,
// K of kind MULTIEXP_SSM) advance in lock step and share every launch of a round:
//   prologue   3K commitments in one pairing chain (table-driven k_miller6), one sync for the K challenges r_k; the
//              powers of every r_k in one launch; a_r and ck_1_r as one G1 and one G2 scaling over all K n elements;
//              agg_c (K segments) and ip_ab with the :133-136 self-check (2K products) on a child stream, joined
//              before the first fold;
//   per round  8K pairing products in one chain, the 2K G1 products of the SSM recursions as two segmented MSMs (one per
//              half: their bases are the upper / lower halves of the arena), one copy of all results, one sync, 2K host
//              challenges, one upload of the fold scalars and one table-driven fold launch for all 7K folds;
//   openings   3K KZG quotients on host threads, the 2K G2 openings and the K G1 openings as two segmented MSMs over the
//              shared SRS, one copy, one sync.
// The vectors live in one arena per vector and recursion kind, instance k at element k n (the instance stride).  Launch
// and synchronisation counts depend on n, not on K.
#pragma once
#include "endo.cuh"

// one entry of the device segment table of ripp_pairing_table_l6 (pairing6.cu's M6Seg): P and Q base pointers
struct M6SegH {
  const void* p;
  const void* q;
};

// page-locked staging grown on demand (the per-round results of K batches outgrow the context's fixed block)
static int pinned_grow(ripp_ctx* ctx, size_t bytes, uint8_t** out) {
  if (ctx->pinned_big_bytes < bytes) {
    if (ctx->pinned_big) CU(cudaFreeHost(ctx->pinned_big));
    ctx->pinned_big = nullptr;
    ctx->pinned_big_bytes = 0;
    CU(cudaHostAlloc((void**)&ctx->pinned_big, bytes, cudaHostAllocDefault));
    ctx->pinned_big_bytes = bytes;
  }
  *out = ctx->pinned_big;
  return RIPP_OK;
}

// fn(i) for i < count (fn must not fail), on host threads when there are at least `grain` items per thread: a thread
// costs tens of microseconds to start, an item of the per-round work (one challenge, two recodings) a few.  Threads that
// cannot be started leave their items to the calling thread.
template <class Fn>
static void host_parallel(size_t count, size_t grain, Fn fn) {
  size_t nt = std::thread::hardware_concurrency();
  if (nt > 32) nt = 32;
  if (nt > count / grain) nt = count / grain;
  std::vector<std::thread> ts;
  size_t started = 0;
  for (size_t t = 1; t < nt; t++) {
    try {
      ts.emplace_back([&, t] {
        for (size_t i = t; i < count; i += nt) fn(i);
      });
      started = t;
    } catch (...) {
      break;
    }
  }
  if (nt < 1) nt = 1;
  for (size_t i = 0; i < count; i++)  // this thread: slot 0, and the slots of threads that did not start
    if (i % nt == 0 || i % nt > started) fn(i);
  for (auto& th : ts) th.join();
}

// r_k^e and r_k^-e for element e < n of segment k (k_fr_powers with r read per segment)
__global__ void k_fr_powers_seg(const Fr* __restrict__ r, const Fr* __restrict__ r_inv, size_t n, size_t total, Fr* __restrict__ pw,
                                Fr* __restrict__ pw_inv) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total) return;
  const size_t k = i / n;
  Fr acc = Fr::one(), acci = Fr::one(), b = r[k], bi = r_inv[k];
  for (size_t e = i - k * n; e; e >>= 1) {
    if (e & 1) {
      acc = acc * b;
      acci = acci * bi;
    }
    b = b * b;
    bi = bi * bi;
  }
  pw[i] = acc;
  pw_inv[i] = acci;
}

// out[k] = in[k stride_words .. + words) for k < count: the base values of the K instances of one arena
__global__ void k_gather_rows(const uint32_t* __restrict__ in, size_t stride_words, uint32_t words, size_t count,
                              uint32_t* __restrict__ out) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= count * words) return;
  const size_t k = t / words;
  out[t] = in[k * stride_words + (t - k * words)];
}

// bytes of one AggregateProof for n = 2^L proofs
static size_t aggregate_proof_len(size_t L) {
  const size_t ab = 8 + L * (6 * 576 + 16) + 96 + 192 + 192 + 96 + 192 + 96;
  const size_t c = 8 + L * (2 * 576 + 2 * 32 + 2 * 96 + 16) + 96 + 32 + 192 + 192;
  return 4 * 576 + 96 + ab + c;
}

static Val val_of(int t, const void* raw) {
  Val v;
  v.t = t;
  memset(v.raw, 0, sizeof(v.raw));
  if (raw) memcpy(v.raw, raw, vt_size(t));
  return v;
}

// count x n at most 2^20 proofs and count at most 2^16 batches: the device workspace is then at most ~41 GB (n = 16 at
// both caps; DESIGN.md §4 gives the per-batch figures)
#define AGG_BATCH_MAX_PROOFS ((size_t)1 << 20)
#define AGG_BATCH_MAX_COUNT ((size_t)1 << 16)

static int agg_batch_check(ripp_ctx* ctx, const void* srs_g1, const void* srs_g2, size_t count, size_t n, const void* a, const void* b,
                           const void* c, uint8_t* proofs_out, size_t proofs_cap, size_t* proof_len) {
  if (!ctx || !srs_g1 || !srs_g2 || !a || !b || !c || !proof_len) return fail(RIPP_ERR_ARG, "null argument");
  if (n == 0 || (n & (n - 1))) return fail(RIPP_ERR_NOT_POW2, "number of proofs must be a power of two");
  if (n < 2) return fail(RIPP_ERR_ARG, "aggregation needs at least two proofs (tipa/mod.rs:199 unwraps the first challenge)");
  if (count == 0) {
    *proof_len = 0;
    return RIPP_OK;
  }
  if (count > AGG_BATCH_MAX_PROOFS / n) return fail(RIPP_ERR_ARG, "batch aggregation: count x n over 2^20 proofs");
  if (count > AGG_BATCH_MAX_COUNT) return fail(RIPP_ERR_ARG, "batch aggregation: more than 2^16 batches");
  size_t L = 0;
  while (((size_t)1 << L) < n) L++;
  const size_t len = aggregate_proof_len(L);
  *proof_len = len;
  if (!proofs_out || proofs_cap / len < count)
    return fail(RIPP_ERR_ARG, "output buffer too small: need " + std::to_string(count * len));
  return RIPP_OK;
}

static int agg_batch(ripp_ctx* ctx, const void* srs_g1, const void* srs_g2, size_t K, size_t n, const void* a_dev, const void* b_dev,
                     const void* c_dev, uint8_t* proofs_out, size_t len) {
  CU(cudaSetDevice(ctx->device));
  cudaStream_t st = ctx->stream;
  size_t L = 0;
  while (((size_t)1 << L) < n) L++;
  const size_t N = K * n;
  auto up = [](size_t x) { return (x + 255) & ~(size_t)255; };
  // ---- arenas: one per vector and recursion kind, instance k at element k n ----
  void* ar;
  const size_t o_abA = 0, o_abB = o_abA + up(N * 96), o_abV = o_abB + up(N * 192), o_abW = o_abV + up(N * 192),
               o_cA = o_abW + up(N * 96), o_cB = o_cA + up(N * 96), o_cV = o_cB + up(N * 32), o_pwi = o_cV + up(N * 192),
               ar_bytes = o_pwi + up(N * 32);
  OK(scratch(ctx, 42, ar_bytes, &ar));
  char* AR = (char*)ar;
  char *abA = AR + o_abA, *abB = AR + o_abB, *abV = AR + o_abV, *abW = AR + o_abW, *cA = AR + o_cA, *cB = AR + o_cB, *cV = AR + o_cV;
  Fr* pwi = (Fr*)(AR + o_pwi);
  // ---- workspace: segment tables of every stage, results, fold scalar records ----
  const size_t nseg_all = 5 * K + 8 * K * L;
  const size_t rec_bytes = 4 * K * sizeof(EndoBits) + K * sizeof(Fr);
  void* ws;
  const size_t o_segs = 0, o_com = o_segs + up(nseg_all * sizeof(M6SegH)), o_ip = o_com + up(3 * K * 576), o_aggc = o_ip + up(2 * K * 576),
               o_res = o_aggc + up(K * 96), o_rec = o_res + up(8 * K * 576 + 2 * K * 96), o_r = o_rec + up(rec_bytes),
               o_open = o_r + up(2 * K * 32), ws_bytes = o_open + up(2 * K * 192 + K * 96);
  OK(scratch(ctx, 41, ws_bytes, &ws));
  char* WS = (char*)ws;
  // ---- page-locked staging: results at the front, uploads behind them ----
  const size_t pres = K * (8 * 576 + 2 * 96), pin_bytes = up(pres) + up(rec_bytes > 2 * K * 32 ? rec_bytes : 2 * K * 32);
  uint8_t* pin;
  OK(pinned_grow(ctx, pin_bytes, &pin));
  uint8_t* pup = pin + up(pres);
  ripp_ctx* kid = ripp_child(ctx, 3);
  ripp_ctx* mk = ripp_child(ctx, 0);
  if (!kid || !mk) return fail(RIPP_ERR_CUDA, "child context");

  // ---- segment tables of all stages, uploaded once ----
  {
    std::vector<M6SegH> segs(nseg_all);
    size_t s = 0;
    auto put = [&](const void* p, const void* q) { segs[s++] = M6SegH{p, q}; };
    const char* ck1 = cV;  // instance 0 of the replicated key before any fold
    const char* ck2 = abW;
    for (size_t k = 0; k < K; k++) {  // :100-102 com_a = IP(a, ck_1), com_b = IP(ck_2, b), com_c = IP(c, ck_1)
      put((const char*)a_dev + k * n * 96, ck1);
      put(ck2, (const char*)b_dev + k * n * 192);
      put((const char*)c_dev + k * n * 96, ck1);
    }
    for (size_t k = 0; k < K; k++) {  // :124 ip_ab = IP(a_r, b), :133-136 IP(a_r, ck_1_r)
      put(abA + k * n * 96, abB + k * n * 192);
      put(abA + k * n * 96, abV + k * n * 192);
    }
    for (size_t h = n / 2; h >= 1; h /= 2) {
      // gipa.rs:209-231 -- com_1 = (IP(A_R, v_L), IP(w_R, B_L), IP(A_R, B_L)); com_2 = (IP(A_L, v_R), IP(w_L, B_R), IP(A_L, B_R))
      for (size_t k = 0; k < K; k++) {
        const char *A = abA + k * n * 96, *B = abB + k * n * 192, *V = abV + k * n * 192, *W = abW + k * n * 96;
        put(A + h * 96, V);
        put(W + h * 96, B);
        put(A + h * 96, B);
        put(A, V + h * 192);
        put(W, B + h * 192);
        put(A, B + h * 192);
      }
      for (size_t k = 0; k < K; k++) {  // the SSM recursion's pairing products IP(A_R, v_L), IP(A_L, v_R)
        const char *A = cA + k * n * 96, *V = cV + k * n * 192;
        put(A + h * 96, V);
        put(A, V + h * 192);
      }
    }
    CU(cudaMemcpyAsync(WS + o_segs, segs.data(), nseg_all * sizeof(M6SegH), cudaMemcpyHostToDevice, st));
  }
  const M6SegH* segs_dev = (const M6SegH*)(WS + o_segs);

  // ---- prologue ----
  double t0 = now_ms();
  const unsigned nb = (unsigned)((n + 127) / 128);
  // :98 commitment keys = even SRS powers, gathered once and replicated for every instance
  k_gather_stride2<G2Aff><<<nb, 128, 0, st>>>((const G2Aff*)srs_g2, n, (G2Aff*)cV);
  LAUNCHED(ctx);
  k_gather_stride2<G1Aff><<<nb, 128, 0, st>>>((const G1Aff*)srs_g1, n, (G1Aff*)abW);
  LAUNCHED(ctx);
  for (size_t have = n; have < N; have *= 2) {
    const size_t m = have < N - have ? have : N - have;
    CU(cudaMemcpyAsync(cV + have * 192, cV, m * 192, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemcpyAsync(abW + have * 96, abW, m * 96, cudaMemcpyDeviceToDevice, st));
  }
  OK(ripp_pairing_table_l6(ctx, segs_dev, 3 * K, n, WS + o_com, 44));
  CU(cudaMemcpyAsync(pin, WS + o_com, 3 * K * 576, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  std::vector<Val> com(3 * K);
  for (size_t i = 0; i < 3 * K; i++) com[i] = val_of(VT_GT, pin + i * 576);
  // :105-116 r_k
  std::vector<Fr> r(K), r_inv(K);
  host_parallel(K, 64, [&](size_t k) {
    Bytes parts;
    for (int i = 0; i < 3; i++) put_val(parts, com[3 * k + i]);
    r[k] = challenge_from_random_bytes(parts);
    r_inv[k] = r[k].inv();
  });
  memcpy(pup, r.data(), K * 32);
  memcpy(pup + K * 32, r_inv.data(), K * 32);
  CU(cudaMemcpyAsync(WS + o_r, pup, 2 * K * 32, cudaMemcpyHostToDevice, st));
  // :118-131 r_vec (into the SSM recursion's right message), a_r = a * r^i, ck_1_r = ck_1 * r^-i
  k_fr_powers_seg<<<(unsigned)((N + 127) / 128), 128, 0, st>>>((const Fr*)(WS + o_r), (const Fr*)(WS + o_r) + K, n, N, (Fr*)cB, pwi);
  LAUNCHED(ctx);
  OK(ripp_g1_scale_dev(ctx, a_dev, cB, N, abA));
  OK(ripp_g2_scale_dev(ctx, cV, pwi, N, abV));
  CU(cudaMemcpyAsync(abB, b_dev, N * 192, cudaMemcpyDeviceToDevice, st));
  CU(cudaMemcpyAsync(cA, c_dev, N * 96, cudaMemcpyDeviceToDevice, st));
  // :124, :133-136 and :125 agg_c = MSM(c, r_vec): on a child stream, overlapping the first round's products; joined
  // before the first fold overwrites their inputs
  OK(ripp_fork(ctx, kid));
  OK(ripp_pairing_table_l6(kid, segs_dev + 3 * K, 2 * K, n, WS + o_ip, 44));
  OK(ripp_msm_batch_internal(kid, 1, c_dev, n, cB, n, n, K, WS + o_aggc));
  if (trace_on()) fprintf(stderr, "[trace] aggregate batch prologue (K = %zu, n = %zu) %.2f ms\n", K, n, now_ms() - t0);

  // ---- rounds in lock step ----
  std::vector<std::vector<Bytes>> steps_ab(K), steps_c(K);  // per instance: serialised rounds, oldest first
  std::vector<std::vector<Fr>> tr_ab(K), tr_c(K);
  std::vector<Fr> cab(K), ciab(K), cc(K), cic(K);
  EndoBits* rec = (EndoBits*)pup;  // [G1 c_ab][G1 c_c][G2 c_ab^-1][G2 c_c^-1] then Fr c_c^-1
  Fr* rec_fr = (Fr*)(rec + 4 * K);
  const char* rec_dev = WS + o_rec;
  const Fr zero = Fr::zero();
  char* res = WS + o_res;
  size_t round = 0;
  for (size_t h = n / 2; h >= 1; h /= 2, round++) {
    double t_r0 = now_ms();
    // the 2K G1 products IP(A_R, B_L), IP(A_L, B_R) of the SSM recursions on a child stream
    OK(ripp_fork(ctx, mk));
    OK(ripp_msm_batch_internal(mk, 1, cA + h * 96, n, cB, n, h, K, res + 8 * K * 576));
    OK(ripp_msm_batch_internal(mk, 1, cA, n, (const Fr*)cB + h, n, h, K, res + 8 * K * 576 + K * 96));
    OK(ripp_pairing_table_l6(ctx, segs_dev + 5 * K + round * 8 * K, 8 * K, h, res, 44));
    OK(ripp_join(ctx, mk));
    CU(cudaMemcpyAsync(pin, res, 8 * K * 576 + 2 * K * 96, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    // gipa.rs:235-258 -- Fiat-Shamir challenges, and the fold scalars' recodings
    host_parallel(2 * K, 64, [&](size_t i) {
      Val v[6];
      Bytes chunk;
      Fr c, ci;
      if (i < K) {
        const size_t k = i;
        for (int j = 0; j < 6; j++) v[j] = val_of(VT_GT, pin + (6 * k + j) * 576);
        gipa_challenge(tr_ab[k].empty() ? zero : tr_ab[k].back(), v, &c, &ci);
        cab[k] = c;
        ciab[k] = ci;
        ripp_endo_bits(1, c.v, &rec[k]);
        ripp_endo_bits(2, ci.v, &rec[2 * K + k]);
      } else {
        const size_t k = i - K;
        const uint8_t* g1 = pin + 8 * K * 576;
        v[0] = val_of(VT_GT, pin + (6 * K + 2 * k) * 576);
        v[1] = val_of(VT_FR, nullptr);  // SSMPlaceholderCommitment
        v[2] = val_of(VT_G1, g1 + k * 96);
        v[3] = val_of(VT_GT, pin + (6 * K + 2 * k + 1) * 576);
        v[4] = val_of(VT_FR, nullptr);
        v[5] = val_of(VT_G1, g1 + (K + k) * 96);
        gipa_challenge(tr_c[k].empty() ? zero : tr_c[k].back(), v, &c, &ci);
        cc[k] = c;
        cic[k] = ci;
        ripp_endo_bits(1, c.v, &rec[K + k]);
        ripp_endo_bits(2, ci.v, &rec[3 * K + k]);
        rec_fr[k] = ci;
      }
      for (int j = 0; j < 6; j++) {
        if (j % 3 == 2) put_u64_le(chunk, 1);
        put_val(chunk, v[j]);
      }
      (i < K ? steps_ab[i] : steps_c[i - K]).push_back(std::move(chunk));
    });
    for (size_t k = 0; k < K; k++) {
      tr_ab[k].push_back(cab[k]);
      tr_c[k].push_back(cc[k]);
    }
    if (round == 0) OK(ripp_join(ctx, kid));  // ip_ab, the self-check and agg_c read the arena
    // gipa.rs:261-291 -- A <- A_R c + A_L, B <- B_R c^-1 + B_L, v <- v_R c^-1 + v_L, w <- w_R c + w_L: one table
    CU(cudaMemcpyAsync(WS + o_rec, pup, rec_bytes, cudaMemcpyHostToDevice, st));
    FoldTable ft;
    memset(&ft, 0, sizeof(ft));
    ft.K = (uint32_t)K;
    ft.n = (uint32_t)h;
    const EndoBits* rd = (const EndoBits*)rec_dev;
    ft.ngroups[0] = 3;  // G1: A (c), w (c) of the pairing recursion, A (c) of the SSM recursion
    ft.base[0][0] = abA, ft.base[0][1] = abW, ft.base[0][2] = cA;
    ft.sc[0][0] = rd, ft.sc[0][1] = rd, ft.sc[0][2] = rd + K;
    ft.ngroups[1] = 3;  // G2: B (c^-1), v (c^-1) of the pairing recursion, v (c^-1) of the SSM recursion
    ft.base[1][0] = abB, ft.base[1][1] = abV, ft.base[1][2] = cV;
    ft.sc[1][0] = rd + 2 * K, ft.sc[1][1] = rd + 2 * K, ft.sc[1][2] = rd + 3 * K;
    ft.ngroups[2] = 1;  // Fr: B (c^-1) of the SSM recursion
    ft.base[2][0] = cB;
    ft.sc[2][0] = rd + 4 * K;
    for (int g = 0; g < 3; g++) {
      ft.stride[0][g] = n * 96;
      ft.stride[1][g] = n * 192;
    }
    ft.stride[2][0] = n * 32;
    OK(ripp_fold_table_internal(ctx, ft));
    if (trace_on()) fprintf(stderr, "[trace] aggregate batch round n' = %zu %.2f ms\n", h, now_ms() - t_r0);
  }

  // ---- base values, ip_ab, the self-check, agg_c: one copy each kind, one sync ----
  double t_o0 = now_ms();
  struct Base {
    const char* src;
    size_t esz;
  };
  const Base bases[7] = {{abA, 96}, {abB, 192}, {abV, 192}, {abW, 96}, {cA, 96}, {cB, 32}, {cV, 192}};
  // element 0 of every instance, gathered into the (now free) round results area, then one copy
  size_t off[8];
  off[0] = 0;
  for (int i = 0; i < 7; i++) {
    const uint32_t words = (uint32_t)(bases[i].esz / 4);
    k_gather_rows<<<(unsigned)((K * words + 127) / 128), 128, 0, st>>>((const uint32_t*)bases[i].src, n * words, words, K,
                                                                      (uint32_t*)(res + off[i]));
    LAUNCHED(ctx);
    off[i + 1] = off[i] + K * bases[i].esz;
  }
  CU(cudaMemcpyAsync(pin, res, off[7], cudaMemcpyDeviceToHost, st));
  // ip_ab / self-check products and agg_c in one copy (o_aggc follows o_ip); 2144 K bytes in all, within the 4800 K of
  // the results area
  CU(cudaMemcpyAsync(pin + off[7], WS + o_ip, (o_aggc - o_ip) + K * 96, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  const uint8_t* ipres = pin + off[7];
  const uint8_t* aggc = ipres + (o_aggc - o_ip);
  auto base_val = [&](int i, int t, size_t k) { return val_of(t, pin + off[i] + k * bases[i].esz); };
  for (size_t k = 0; k < K; k++) {
    Bytes x, y;
    put_val(x, com[3 * k]);
    put_val(y, val_of(VT_GT, ipres + (2 * k + 1) * 576));
    if (x != y)
      return fail(RIPP_ERR_INNER_PRODUCT,
                  "batch " + std::to_string(k) + ": com_a != IP(a_r, ck_1_r) (groth16_aggregation.rs:133-136)");
  }
  // ---- KZG openings (tipa/mod.rs:195-209, 304-337; structured_scalar_message.rs:238-251) ----
  const size_t n_srs = 2 * n - 1;
  void* qd;
  OK(scratch(ctx, 43, 3 * K * n_srs * sizeof(Fr) + 256, &qd));
  std::vector<Fr> q(3 * K * n_srs);
  host_parallel(2 * K, n >= 256 ? 1 : 16, [&](size_t i) {
    const bool ab = i < K;
    const size_t k = ab ? i : i - K;
    const std::vector<Fr>& tr = ab ? tr_ab[k] : tr_c[k];
    std::vector<Fr> rev(tr.rbegin(), tr.rend()), tinv(rev.size());
    for (size_t j = 0; j < rev.size(); j++) tinv[j] = rev[j].inv();
    Bytes parts;
    put_fr(parts, rev[0]);
    put_val(parts, base_val(ab ? 2 : 6, VT_G2, k));
    if (ab) put_val(parts, base_val(3, VT_G1, k));
    const Fr z = challenge_from_random_bytes(parts);
    std::vector<Fr> qa = kzg_quotient(tinv, ab ? r_inv[k] : Fr::one(), z, n_srs);  // the SSM variant opens with shift 1
    memcpy(&q[i * n_srs], qa.data(), n_srs * sizeof(Fr));
    if (ab) {
      std::vector<Fr> qb = kzg_quotient(rev, Fr::one(), z, n_srs);
      memcpy(&q[(2 * K + k) * n_srs], qb.data(), n_srs * sizeof(Fr));
    }
  });
  if (trace_on()) fprintf(stderr, "[trace] aggregate batch quotients (host) %.2f ms\n", now_ms() - t_o0);
  CU(cudaMemcpyAsync(qd, q.data(), q.size() * sizeof(Fr), cudaMemcpyHostToDevice, st));
  char* op = WS + o_open;
  OK(ripp_fork(ctx, mk));
  OK(ripp_msm_batch_internal(mk, 1, srs_g1, 0, (const Fr*)qd + 2 * K * n_srs, n_srs, n_srs, K, op + 2 * K * 192));
  OK(ripp_msm_batch_internal(ctx, 2, srs_g2, 0, qd, n_srs, n_srs, 2 * K, op));
  OK(ripp_join(ctx, mk));
  // into the upload area (K (4 x 168 + 32) bytes >= 480 K): the results area still holds the base values
  uint8_t* openings = pup;
  CU(cudaMemcpyAsync(openings, op, 2 * K * 192 + K * 96, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  if (trace_on()) fprintf(stderr, "[trace] aggregate batch openings %.2f ms\n", now_ms() - t_o0);

  // ---- AggregateProof { com_a, com_b, com_c, ip_ab, agg_c, tipa_proof_ab, tipa_proof_c } (:58-66) ----
  std::vector<int> bad(K, 0);
  host_parallel(K, 16, [&](size_t k) {
    Bytes out;
    out.reserve(len);
    for (int i = 0; i < 3; i++) put_val(out, com[3 * k + i]);
    put_val(out, val_of(VT_GT, ipres + 2 * k * 576));
    put_val(out, val_of(VT_G1, aggc + k * 96));
    // TIPAProof of the pairing recursion: GIPAProof (rounds newest first, r_base), final ck, the two openings
    put_u64_le(out, L);
    for (size_t i = L; i-- > 0;) out.insert(out.end(), steps_ab[k][i].begin(), steps_ab[k][i].end());
    put_val(out, base_val(0, VT_G1, k));
    put_val(out, base_val(1, VT_G2, k));
    put_val(out, base_val(2, VT_G2, k));
    put_val(out, base_val(3, VT_G1, k));
    put_val(out, val_of(VT_G2, openings + k * 192));
    put_val(out, val_of(VT_G1, openings + 2 * K * 192 + k * 96));
    // TIPAWithSSMProof of the C recursion
    put_u64_le(out, L);
    for (size_t i = L; i-- > 0;) out.insert(out.end(), steps_c[k][i].begin(), steps_c[k][i].end());
    put_val(out, base_val(4, VT_G1, k));
    put_val(out, base_val(5, VT_FR, k));
    put_val(out, base_val(6, VT_G2, k));
    put_val(out, val_of(VT_G2, openings + (K + k) * 192));
    if (out.size() != len) {
      bad[k] = 1;
      return;
    }
    memcpy(proofs_out + k * len, out.data(), len);
  });
  for (size_t k = 0; k < K; k++)
    if (bad[k]) return fail(RIPP_ERR_CUDA, "batch " + std::to_string(k) + ": proof length differs from the layout");
  return RIPP_OK;
}

extern "C" int ripp_tipp_aggregate_batch_dev(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, size_t count, size_t n,
                                             const void* a_dev, const void* b_dev, const void* c_dev, uint8_t* proofs_out,
                                             size_t proofs_cap, size_t* proof_len) {
  OK(agg_batch_check(ctx, srs_g1_dev, srs_g2_dev, count, n, a_dev, b_dev, c_dev, proofs_out, proofs_cap, proof_len));
  if (count == 0) return RIPP_OK;
  return agg_batch(ctx, srs_g1_dev, srs_g2_dev, count, n, a_dev, b_dev, c_dev, proofs_out, *proof_len);
}

extern "C" int ripp_tipp_aggregate_batch(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, size_t count, size_t n,
                                         const void* a_host, const void* b_host, const void* c_host, uint8_t* proofs_out,
                                         size_t proofs_cap, size_t* proof_len) {
  OK(agg_batch_check(ctx, srs_g1_dev, srs_g2_dev, count, n, a_host, b_host, c_host, proofs_out, proofs_cap, proof_len));
  if (count == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  const size_t N = count * n;
  void* d;
  OK(scratch(ctx, 46, N * (96 + 192 + 96) + 1024, &d));
  char* p = (char*)d;
  CU(cudaMemcpyAsync(p, a_host, N * 96, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(p + N * 96, c_host, N * 96, cudaMemcpyHostToDevice, ctx->stream));
  CU(cudaMemcpyAsync(p + N * 192, b_host, N * 192, cudaMemcpyHostToDevice, ctx->stream));
  return agg_batch(ctx, srs_g1_dev, srs_g2_dev, count, n, p, p + N * 192, p + N * 96, proofs_out, *proof_len);
}
