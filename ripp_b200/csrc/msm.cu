// Variable-base MSM (Pippenger) over G1/G2, uniform-scalar folds and Fr vector ops.
//
// Replaces (SURVEY.md §8a): `G::msm(normalize_batch(L), R)` of MultiexponentiationInnerProduct
// (inner_products/src/lib.rs:123-142), PedersenCommitment::commit (pedersen/mod.rs:24-26), the KZG
// opening MSMs (tipa/mod.rs:333-334), and the "rescale" maps of GIPA/SIPP (gipa.rs:261-291,
// sipp/src/lib.rs:87-100; scalar-mul primitive `mul_helper`, ip_proofs/src/lib.rs:15-19).
#include <optional>

#include "common.cuh"
#include "x3.cuh"
#include "xt.cuh"

static bool use_endo() {
  static const bool v = [] {
    const char* e = getenv("RIPP_B200_FOLD");  // "plain" = no endomorphism (A/B runs)
    return !(e && strcmp(e, "plain") == 0);
  }();
  return v;
}

// ------------------------------------------------------------------------------------------------
// MSM
// ------------------------------------------------------------------------------------------------
struct MsmPlan {
  int c;       // window bits
  int nw;      // windows
  uint32_t B;  // buckets per window: 2^(c-1), slot i holds the points whose SIGNED digit has magnitude i + 1
  uint32_t L;  // buckets per reduction chunk
  uint32_t T;  // chunks per window
};

#define MSM_SMALL_N ((size_t)1 << 16)
// seg: one segment of a segmented MSM (nseg > 1).  A short segment then takes its window from its own length, down to
// c = 2 + 1, instead of the single MSM's floor of 6 + 1: the floor's nw x 64 buckets and 2 nw x 32 partials (~370 KB for
// a G2 segment) would dwarf a segment of a few points, and a batch of 2^20 such segments would not fit the GPU.  The
// window width does not change the result.
static MsmPlan msm_plan(size_t n, int bits = 255, bool seg = false) {
  int lg = 0;
  while (((size_t)2 << lg) <= n) lg++;
  MsmPlan p;
  // ~32 points per bucket: long enough that the Poisson spread of bucket sizes does not idle most of a
  // warp (at 4 per bucket a warp runs at max/mean ~ 2.5x), short enough for the small MSMs of late rounds
  static const int shift = [] {  // RIPP_B200_MSM_SHIFT: log2 of the target points per bucket (tuning runs)
    const char* e = getenv("RIPP_B200_MSM_SHIFT");
    return e ? atoi(e) : 5;
  }();
  // short inputs (the KZG openings and the MSM-type products of the GIPA rounds) are latency chains on an empty GPU:
  // ~4 points per bucket keeps the per-bucket chain short; below 2^6 points the window only sets the Horner tail
  p.c = lg - (n <= MSM_SMALL_N ? 2 : shift);
  const int c_min = n <= MSM_SMALL_N ? (seg ? 2 : 6) : 4;
  if (p.c < c_min) p.c = c_min;
  if (p.c > 15) p.c = 15;
  // signed digits d_w in (-2^(c-1), 2^(c-1)] (the negative of a point is free): half the buckets of an unsigned window
  // for the same c, i.e. one more bit per window at equal bucket count.  The recoding may carry out of the top digit:
  // one more bit of room.
  p.c += 1;
  p.nw = (bits + 1 + p.c - 1) / p.c;
  p.B = 1u << (p.c - 1);
  p.L = p.B / 256;  // short chunks: the running-sum chains are latency, not throughput
  if (p.L < 2) p.L = 2;
  if (p.L > 8) p.L = 8;
  p.T = p.B / p.L;
  return p;
}

__device__ __forceinline__ uint32_t msm_digit(const uint32_t* s, int w, int c) {
  int o = w * c;
  int wi = o >> 5, sh = o & 31;
  uint64_t v = s[wi];
  if (wi + 1 < 8) v |= (uint64_t)s[wi + 1] << 32;
  return (uint32_t)(v >> sh) & ((1u << c) - 1);
}

// signed recoding, window by window with a running carry: returns the magnitude (0 .. 2^(c-1)) and the sign
__device__ __forceinline__ uint32_t msm_sdigit(const uint32_t* s, int w, int c, uint32_t& carry, bool& neg) {
  uint32_t raw = (w * c < 256 ? msm_digit(s, w, c) : 0u) + carry;  // <= 2^c
  const uint32_t half = 1u << (c - 1);
  neg = raw > half;
  carry = neg ? 1u : 0u;
  return neg ? (1u << c) - raw : raw;
}

// canonical scalars + per-(segment, window, bucket) histogram; n = nseg x seg_n scalars, segment s's at sc + s sc_stride
// (SEG = false: one segment, seg_n = n; the single MSM's code)
template <bool SEG>
__global__ void k_msm_prepare(const Fr* __restrict__ sc, size_t n, Fr* __restrict__ canon, uint32_t* __restrict__ counts,
                              int c, int nw, int is_mont, size_t seg_n, size_t sc_stride) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t seg = SEG ? i / seg_n : 0;
  const Fr v = sc[seg * sc_stride + (i - seg * seg_n)];
  Fr s = is_mont ? v.from_mont() : v;
  canon[i] = s;
  uint32_t B = 1u << (c - 1), carry = 0;
  for (int w = 0; w < nw; w++) {
    bool neg;
    uint32_t d = msm_sdigit(s.v, w, c, carry, neg);
    if (d) atomicAdd(&counts[(seg * nw + w) * B + d - 1], 1u);
  }
}

// Buckets with more than MSM_FAT points (the top window of any 255-bit scalar set is always skewed:
// it has few significant bits, hence few, huge buckets) are split into chunks of MSM_FAT_CHUNK points
// summed by whole blocks; everything else is one thread per bucket.
#define MSM_FAT 96u
#define MSM_FAT_CHUNK 2048u
struct FatItem {
  uint32_t bucket;  // w * B + digit
  uint32_t chunk;   // chunk index within the bucket
};
struct FatBucket {
  uint32_t bucket, first_item, nchunks;
};

// exclusive scan of counts within each window (one block per window; the nseg x nw windows of a segmented MSM in
// segment-major order) -> offsets into idx[w*n ..], n = points per segment
__global__ void k_msm_scan(const uint32_t* __restrict__ counts, uint32_t* __restrict__ offsets,
                           uint32_t* __restrict__ cursor, uint32_t B, size_t n, uint32_t* __restrict__ fat_counters,
                           FatItem* __restrict__ items, FatBucket* __restrict__ fats, uint32_t max_items,
                           uint32_t fat_threshold) {
  __shared__ uint32_t part[256];
  int w = blockIdx.x;
  uint32_t per = (B + 255) / 256;
  uint32_t lo = threadIdx.x * per, hi = lo + per < B ? lo + per : B;
  uint32_t s = 0;
  for (uint32_t j = lo; j < hi; j++) s += counts[(size_t)w * B + j];
  part[threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    uint32_t run = 0;
    for (int t = 0; t < 256; t++) {
      uint32_t v = part[t];
      part[t] = run;
      run += v;
    }
  }
  __syncthreads();
  uint32_t run = part[threadIdx.x] + (uint32_t)((size_t)w * n);
  for (uint32_t j = lo; j < hi; j++) {
    uint32_t cnt = counts[(size_t)w * B + j];
    offsets[(size_t)w * B + j] = run;
    cursor[(size_t)w * B + j] = run;
    run += cnt;
    if (cnt > fat_threshold) {
      uint32_t nch = (cnt + MSM_FAT_CHUNK - 1) / MSM_FAT_CHUNK;
      uint32_t first = atomicAdd(&fat_counters[0], nch);
      uint32_t fb = atomicAdd(&fat_counters[1], 1u);
      if (first + nch <= max_items) {
        fats[fb] = FatBucket{(uint32_t)((size_t)w * B + j), first, nch};
        for (uint32_t k = 0; k < nch; k++) items[first + k] = FatItem{(uint32_t)((size_t)w * B + j), k};
      }
    }
  }
}

// index entries are positions within the segment (the segment's bases are found from the bucket id)
template <bool SEG>
__global__ void k_msm_scatter(const Fr* __restrict__ canon, size_t n, uint32_t* __restrict__ cursor,
                              uint32_t* __restrict__ idx, int c, int nw, size_t seg_n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const size_t seg = SEG ? i / seg_n : 0;
  Fr s = canon[i];
  uint32_t B = 1u << (c - 1), carry = 0;
  for (int w = 0; w < nw; w++) {
    bool neg;
    uint32_t d = msm_sdigit(s.v, w, c, carry, neg);
    if (d)  // bit 31: subtract
      idx[atomicAdd(&cursor[(seg * nw + w) * B + d - 1], 1u)] = (uint32_t)(i - seg * seg_n) | (neg ? 0x80000000u : 0u);
  }
}

// ---- buckets sorted by size: a warp of the accumulate kernel then walks 32 buckets of (nearly) equal length ------
// counting sort of the non-empty, non-fat bucket ids by descending point count (bins 1 .. fat_threshold)
__global__ void k_msm_size_hist(const uint32_t* __restrict__ counts, size_t total, uint32_t fat_threshold, uint32_t* __restrict__ hist) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  uint32_t cnt = counts[t];
  if (cnt && cnt <= fat_threshold) atomicAdd(&hist[cnt], 1u);
}
// hist[s] -> start of size s in `order` (largest first); hist[0] <- number of sorted buckets
__global__ void k_msm_size_scan(uint32_t* __restrict__ hist, uint32_t fat_threshold) {
  if (threadIdx.x || blockIdx.x) return;
  uint32_t run = 0;
  for (uint32_t sz = fat_threshold; sz >= 1; sz--) {
    uint32_t v = hist[sz];
    hist[sz] = run;
    run += v;
  }
  hist[0] = run;
}
__global__ void k_msm_size_scatter(const uint32_t* __restrict__ counts, size_t total, uint32_t fat_threshold,
                                   uint32_t* __restrict__ hist, uint32_t* __restrict__ order) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  uint32_t cnt = counts[t];
  if (cnt && cnt <= fat_threshold) order[atomicAdd(&hist[cnt], 1u)] = (uint32_t)t;
}

// one thread per non-empty bucket, in order of decreasing size (`order`, n_sorted = *n_sorted_dev entries): sum of the
// bucket's points; bit 31 of an index entry = the point enters negated (signed window digits).  Bucket b belongs to
// segment b / seg_buckets, whose bases start at bases + segment * bases_stride.
template <class F, bool SEG>
__global__ void __launch_bounds__(128) k_msm_accumulate(const Aff<F>* __restrict__ bases, const uint32_t* __restrict__ idx,
                                                        const uint32_t* __restrict__ offsets,
                                                        const uint32_t* __restrict__ counts, Jac<F>* __restrict__ buckets,
                                                        const uint32_t* __restrict__ order, const uint32_t* __restrict__ n_sorted_dev,
                                                        uint32_t seg_buckets, size_t bases_stride) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= *n_sorted_dev) return;
  const uint32_t b = order[t];
  if (SEG) bases += (size_t)(b / seg_buckets) * bases_stride;
  uint32_t start = offsets[b], cnt = counts[b];
  Jac<F> acc = Jac<F>::inf();
  for (uint32_t j = 0; j < cnt; j++) {
    uint32_t e = idx[start + j];
    Aff<F> p = bases[e & 0x7fffffffu];
    if (e >> 31) p = p.neg();
    acc = acc.add_mixed(p);
  }
  buckets[b] = acc;
}

// one block per (fat bucket, chunk): strided partial sums, then a shared-memory tree
template <class F, bool SEG>
__global__ void __launch_bounds__(128) k_msm_fat_chunks(const Aff<F>* __restrict__ bases, const uint32_t* __restrict__ idx,
                                                        const uint32_t* __restrict__ offsets,
                                                        const uint32_t* __restrict__ counts,
                                                        const uint32_t* __restrict__ fat_counters,
                                                        const FatItem* __restrict__ items, Jac<F>* __restrict__ partials,
                                                        uint32_t seg_buckets, size_t bases_stride) {
  __shared__ Jac<F> sh[128];
  for (uint32_t it = blockIdx.x; it < fat_counters[0]; it += gridDim.x) {
    FatItem w = items[it];
    const Aff<F>* bs = SEG ? bases + (size_t)(w.bucket / seg_buckets) * bases_stride : bases;
    uint32_t start = offsets[w.bucket] + w.chunk * MSM_FAT_CHUNK;
    uint32_t end = offsets[w.bucket] + counts[w.bucket];
    if (end > start + MSM_FAT_CHUNK) end = start + MSM_FAT_CHUNK;
    Jac<F> acc = Jac<F>::inf();
    for (uint32_t j = start + threadIdx.x; j < end; j += 128) {
      uint32_t e = idx[j];
      Aff<F> p = bs[e & 0x7fffffffu];
      if (e >> 31) p = p.neg();
      acc = acc.add_mixed(p);
    }
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int s = 64; s >= 1; s >>= 1) {
      if ((int)threadIdx.x < s) sh[threadIdx.x] = sh[threadIdx.x].add(sh[threadIdx.x + s]);
      __syncthreads();
    }
    if (threadIdx.x == 0) partials[it] = sh[0];
    __syncthreads();
  }
}
// one block per fat bucket: strided sums of its chunk partials, then a shared-memory tree (a top window of a 128-bit
// digit set holds one or two buckets of ~10^5 points = ~85 chunks: summed by ONE thread that was 0.83 ms of a 6.4 ms MSM)
template <class F>
__global__ void __launch_bounds__(64) k_msm_fat_combine(const uint32_t* __restrict__ fat_counters, const FatBucket* __restrict__ fats,
                                                        const Jac<F>* __restrict__ partials, Jac<F>* __restrict__ buckets) {
  __shared__ Jac<F> sh[64];
  for (uint32_t t = blockIdx.x; t < fat_counters[1]; t += gridDim.x) {
    FatBucket fb = fats[t];
    Jac<F> acc = Jac<F>::inf();
    for (uint32_t k = threadIdx.x; k < fb.nchunks; k += 64) acc = acc.add(partials[fb.first_item + k]);
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int st = 32; st >= 1; st >>= 1) {
      if ((int)threadIdx.x < st) sh[threadIdx.x] = sh[threadIdx.x].add(sh[threadIdx.x + st]);
      __syncthreads();
    }
    if (threadIdx.x == 0) buckets[fb.bucket] = sh[0];
    __syncthreads();
  }
}

// one thread per (window, chunk of L buckets): sum_b b * bucket[b] restricted to the chunk
template <class F>
__global__ void __launch_bounds__(128) k_msm_bucket_reduce(const Jac<F>* __restrict__ buckets, uint32_t B, uint32_t L,
                                                           uint32_t T, Jac<F>* __restrict__ partials, size_t total) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  uint32_t w = (uint32_t)(t / T), ch = (uint32_t)(t % T);
  uint32_t j0 = ch * L;  // chunk covers buckets j0 .. j0+L-1 (bucket 0 is empty)
  Jac<F> run = Jac<F>::inf(), acc = Jac<F>::inf();
  for (uint32_t b = L; b-- > 0;) {
    run = run.add(buckets[(size_t)w * B + j0 + b]);
    if (b > 0) acc = acc.add(run);
  }
  // acc = sum_b b_local * bucket, run = sum bucket; slot j0 + b_local carries weight j0 + b_local + 1: add (j0 + 1) run
  if (!run.is_inf()) {
    const uint32_t wgt = j0 + 1;
    Jac<F> m = Jac<F>::inf();
    for (int bit = 31 - __clz(wgt); bit >= 0; bit--) {
      m = m.dbl();
      if ((wgt >> bit) & 1) m = m.add(run);
    }
    acc = acc.add(m);
  }
  partials[t] = acc;
}

// segmented sum: out[w][t] = sum in[w][t*R .. min(T, t*R+R))
template <class F>
__global__ void __launch_bounds__(128) k_jac_reduce(const Jac<F>* __restrict__ in, uint32_t T, uint32_t R, uint32_t To,
                                                    Jac<F>* __restrict__ out, size_t total) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  uint32_t w = (uint32_t)(t / To), k = (uint32_t)(t % To);
  uint32_t lo = k * R, hi = lo + R < T ? lo + R : T;
  Jac<F> acc = in[(size_t)w * T + lo];
  for (uint32_t j = lo + 1; j < hi; j++) acc = acc.add(in[(size_t)w * T + j]);
  out[t] = acc;
}

// out[w] = sum_t in[w][t], t < T: one block per window
template <class F> struct WSUM_THREADS { static constexpr int N = 256; };
template <> struct WSUM_THREADS<Fq2> { static constexpr int N = 128; };  // 128 x 288 B of shared memory
template <class F>
__global__ void __launch_bounds__(WSUM_THREADS<F>::N) k_msm_window_sum(const Jac<F>* __restrict__ in, uint32_t T, Jac<F>* __restrict__ out) {
  constexpr int NT = WSUM_THREADS<F>::N;
  __shared__ Jac<F> sh[NT];
  const Jac<F>* src = in + (size_t)blockIdx.x * T;
  Jac<F> acc = Jac<F>::inf();
  for (uint32_t t = threadIdx.x; t < T; t += NT) acc = acc.add(src[t]);
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int st = NT / 2; st >= 1; st >>= 1) {
    if ((int)threadIdx.x < st) sh[threadIdx.x] = sh[threadIdx.x].add(sh[threadIdx.x + st]);
    __syncthreads();
  }
  if (threadIdx.x == 0) out[blockIdx.x] = sh[0];
}

// Horner tails: one block per segment, block s reads window sums [s nw, s nw + nw) and writes out[s]
template <class F>
__global__ void k_msm_horner(const Jac<F>* __restrict__ sums, int nw, int c, Aff<F>* __restrict__ out) {
  if (threadIdx.x) return;
  sums += (size_t)blockIdx.x * nw;
  out += blockIdx.x;
  Jac<F> acc = sums[nw - 1];
  for (int w = nw - 2; w >= 0; w--) {
    for (int j = 0; j < c; j++) acc = acc.dbl();
    acc = acc.add(sums[w]);
  }
  *out = acc.to_affine();
}

// RIPP_B200_FOLD = "w3" / "endo" / "plain" forces a fold kernel (A/B runs); default: three-warp teams (x3.cuh) while the
// vector is short enough that the GPU is otherwise empty, one thread per element with the endomorphism above that.
static int fold_mode() {
  static const int v = [] {
    const char* e = getenv("RIPP_B200_FOLD");
    return !e ? 0 : (strcmp(e, "w3") == 0 ? 1 : (strcmp(e, "endo") == 0 ? 2 : (strcmp(e, "plain") == 0 ? 3 : 0)));
  }();
  return v;
}
// 3 warps per 32 elements: the team kernels pay off while the GPU is otherwise empty (RIPP_B200_W3_MAX overrides)
static size_t w3_max_n() {
  static const long v = [] {
    const char* e = getenv("RIPP_B200_W3_MAX");
    return e ? atol(e) : 512L;  // TIPP 2^12: 148.5 ms without teams, 143.1 at 512, 146.2 at 4096 (the early rounds already fill the GPU)
  }();
  return (size_t)v;
}

// Horner tail on one three-warp team (<<<1, 96>>>; all lanes hold the same values)
template <class XF>
__global__ void __maxnreg__(255) k_msm_horner_x3(const Jac<XF>* __restrict__ sums, int nw, int c, Aff<XF>* __restrict__ out) {
  sums += (size_t)blockIdx.x * nw;
  out += blockIdx.x;
  Jac<XF> acc = sums[nw - 1];
  for (int w = nw - 2; w >= 0; w--) {
    for (int j = 0; j < c; j++) acc = x3::Ops<XF>::dbl(acc);
    acc = acc.add(sums[w]);  // uniform data: every thread takes the same branch of the complete addition
  }
  Aff<XF> o = x3::to_affine(acc);
  if (threadIdx.x == 0) *out = o;
}
// Horner tail on lane teams (xt.cuh): phase 1, team w brings window sum w to affine form (one inversion each, all windows
// in parallel) into shared memory; phase 2, the first team of warp 0 walks the (nw - 1) c doublings with mixed additions.
// 115 doublings of a G1 tail: 1.19 ms on a three-warp team (k_msm_horner_x3, CTA barriers) -> lanes of one warp.
template <class F>
__global__ void __launch_bounds__(32 * 9) k_msm_horner_xt(const Jac<F>* __restrict__ sums, int nw, int c, Aff<F>* __restrict__ out) {
  typedef xt::TeamOf<F> TO;
  constexpr int AW = sizeof(Aff<F>) / 4;
  extern __shared__ __align__(16) uint32_t hsm[];
  const int warps = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  sums += (size_t)blockIdx.x * nw;
  out += blockIdx.x;
  uint32_t* aff = hsm;                                        // nw affine window sums
  uint32_t* bus = hsm + ((nw * AW + 3) & ~3);                 // per team: 2 bus buffers
  const int vl = lane % (TO::LANES * TO::PER_WARP), e = vl / TO::LANES;
  xt::Team tm{vl % TO::LANES, bus + (warp * TO::PER_WARP + e) * 2 * TO::BUS_WORDS, 0, nullptr};
  for (int w0 = 0; w0 < nw; w0 += warps * TO::PER_WARP) {  // warp-uniform trip count
    int w = w0 + warp * TO::PER_WARP + e;
    const bool live = w < nw && lane == vl;
    if (w >= nw) w = nw - 1;
    Aff<F> a = xt::to_affine<F>(tm, sums[w]);
    if (live && tm.t == 0) xt::aff_st<F>(aff + w * AW, a);
  }
  __syncthreads();
  if (warp) return;
  Jac<F> acc = Jac<F>::from_affine(xt::aff_ld<F>(aff + (nw - 1) * AW));
#pragma unroll 1
  for (int w = nw - 2; w >= 0; w--) {
#pragma unroll 1
    for (int j = 0; j < c; j++) acc = xt::dbl<F>(tm, acc);
    acc = xt::madd<F>(tm, acc, xt::aff_ld<F>(aff + w * AW));
  }
  Aff<F> o = xt::to_affine<F>(tm, acc);
  if (threadIdx.x == 0) *out = o;
}
template <class F>
static size_t horner_xt_smem(int nw) {
  typedef xt::TeamOf<F> TO;
  int warps = (nw + TO::PER_WARP - 1) / TO::PER_WARP;
  if (warps > 9) warps = 9;
  return (size_t)4 * (((nw * (sizeof(Aff<F>) / 4) + 3) & ~3) + warps * TO::PER_WARP * 2 * TO::BUS_WORDS);
}

template <class F> struct X3Of;
template <> struct X3Of<Fq> { typedef Fq type; };
template <> struct X3Of<Fq2> { typedef x3::Fq2x3 type; };

// sum_i s_i P_i = sum_i sum_t d_{i,t} E^t(P_i): m n points with short (128- / 64-bit) scalars, which cuts the
// Horner tail (the latency floor of every MSM) from 255 to 128 / 64 doublings at the same bucket work
// Segmented (nseg segments of n; segment s at bases + s bases_stride, sc + s sc_stride): segment s expands into the m n
// entries [s m n, s m n + m n) of canon2 and, with bases_stride != 0, of bases2; with bases_stride = 0 (one base vector
// for all segments) only segment 0 writes its m n bases.
template <class F>
__global__ void __launch_bounds__(128) k_msm_endo_expand(const Aff<F>* __restrict__ bases, const Fr* __restrict__ sc, size_t n,
                                                         Aff<F>* __restrict__ bases2, Fr* __restrict__ canon2, int m, size_t nseg,
                                                         size_t bases_stride, size_t sc_stride) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * nseg) return;
  const size_t seg = i / n, e = i - seg * n, o = seg * m * n;
  Fr s = sc[seg * sc_stride + e].from_mont();
  uint32_t digits[4][4];
  int mm;
  endo_digits<sizeof(F) == sizeof(Fq) ? 1 : 2>(s.v, digits, &mm);
  Aff<F> p = bases[seg * bases_stride + e];
  const bool put_bases = bases_stride || seg == 0;
  for (int t = 0; t < m; t++) {
    Fr d = Fr::zero();
    for (int j = 0; j < 4; j++) d.v[j] = digits[t][j];
    if (put_bases) bases2[(bases_stride ? o : 0) + (size_t)t * n + e] = p;
    canon2[o + (size_t)t * n + e] = d;
    if (t + 1 < m) p = endo_map(p);
  }
}

template <class F>
static int msm_core(ripp_ctx* ctx, const Aff<F>* bases, size_t bases_stride, const Fr* sc, size_t sc_stride, size_t n, size_t nseg,
                    Aff<F>* out, int bits, int is_mont);

// out[s] = sum_i sc[s sc_stride + i] bases[s bases_stride + i], i < n, s < nseg (bases_stride 0: one base vector shared
// by all segments).  nseg = 1 is the single MSM.
template <class F>
static int msm_dev(ripp_ctx* ctx, const Aff<F>* bases, const Fr* sc, size_t n, Aff<F>* out, size_t nseg = 1, size_t bases_stride = 0,
                   size_t sc_stride = 0) {
  CU(cudaSetDevice(ctx->device));
  if (n == 0) {
    CU(cudaMemsetAsync(out, 0, nseg * sizeof(Aff<F>), ctx->stream));
    return RIPP_OK;
  }
  if (!use_endo()) return msm_core<F>(ctx, bases, bases_stride, sc, sc_stride, n, nseg, out, 255, 1);
  const int m = sizeof(F) == sizeof(Fq) ? 2 : 4;
  const size_t mn = (size_t)m * n;
  void* ex;
  size_t pts_bytes = ((bases_stride ? nseg : 1) * mn * sizeof(Aff<F>) + 255) & ~(size_t)255;
  OK(scratch(ctx, 16, pts_bytes + nseg * mn * sizeof(Fr) + 256, &ex));
  Aff<F>* bases2 = (Aff<F>*)ex;
  Fr* canon2 = (Fr*)((char*)ex + pts_bytes);
  {
    TimeScope ts_(ctx, RIPP_T_MSM_SORT);
    k_msm_endo_expand<F><<<(unsigned)((nseg * n + 127) / 128), 128, 0, ctx->stream>>>(bases, sc, n, bases2, canon2, m, nseg,
                                                                                    bases_stride, sc_stride);
    LAUNCHED(ctx);
  }
  return msm_core<F>(ctx, bases2, bases_stride ? mn : 0, canon2, mn, mn, nseg, out, m == 2 ? 128 : 64, 0);
}

// Segmented Pippenger: nseg independent MSMs of n points in one pass.  Every phase runs over the nseg x nw windows as one
// set, a bucket keyed by (segment, window, digit); the plan (window width, chunks) is that of ONE segment of n points, so
// a segment gets the buckets its own MSM would have and the launch sequence is that of the single MSM.
template <class F>
static int msm_core(ripp_ctx* ctx, const Aff<F>* bases, size_t bases_stride, const Fr* sc, size_t sc_stride, size_t n, size_t nseg,
                    Aff<F>* out, int bits, int is_mont) {
  MsmPlan p = msm_plan(n, bits, nseg > 1);
  const size_t seg_buckets = (size_t)p.nw * p.B;  // buckets of one segment
  const size_t nw = nseg * p.nw;                  // windows of all segments
  const size_t N = nseg * n;                      // points of all segments
  size_t WB = nw * p.B;
  void *canon, *cnt, *idx, *bkt, *parts;
  OK(scratch(ctx, 4, N * sizeof(Fr), &canon));
  OK(scratch(ctx, 5, 3 * WB * sizeof(uint32_t), &cnt));
  OK(scratch(ctx, 6, nw * n * sizeof(uint32_t), &idx));
  OK(scratch(ctx, 7, WB * sizeof(Jac<F>), &bkt));
  OK(scratch(ctx, 8, 2 * nw * p.T * sizeof(Jac<F>), &parts));
  uint32_t* counts = (uint32_t*)cnt;
  uint32_t* offsets = counts + WB;
  uint32_t* cursor = offsets + WB;
  cudaStream_t st = ctx->stream;
  // fat-bucket bookkeeping: at most nw*n/MSM_FAT fat buckets, nw*(n/CHUNK + n/FAT) chunk items
  const uint32_t fat_min = n <= MSM_SMALL_N ? 16u : MSM_FAT;
  uint32_t max_fat = (uint32_t)(nw * n / fat_min + nw + 1);
  uint32_t max_items = (uint32_t)(nw * n / MSM_FAT_CHUNK + max_fat + 1);
  void* fatbuf;
  OK(scratch(ctx, 15, 64 + (size_t)max_items * (sizeof(FatItem) + sizeof(Jac<F>)) + (size_t)max_fat * sizeof(FatBucket) + 1024, &fatbuf));
  uint32_t* fat_counters = (uint32_t*)fatbuf;
  Jac<F>* fat_partials = (Jac<F>*)((char*)fatbuf + 64);
  FatItem* fat_items = (FatItem*)(fat_partials + max_items);
  FatBucket* fat_buckets = (FatBucket*)(fat_items + max_items);
  std::optional<TimeScope> ts_;  // one accounting scope per kernel group: sort, accumulate, reduce
  ts_.emplace(ctx, RIPP_T_MSM_SORT);
  CU(cudaMemsetAsync(fat_counters, 0, 64, st));
  CU(cudaMemsetAsync(counts, 0, WB * sizeof(uint32_t), st));
  const bool seg = nseg > 1;
  (seg ? k_msm_prepare<true> : k_msm_prepare<false>)<<<(unsigned)((N + 127) / 128), 128, 0, st>>>(sc, N, (Fr*)canon, counts, p.c, p.nw,
                                                                                                  is_mont, n, sc_stride);
  LAUNCHED(ctx);
  // "fat" = far above the mean bucket size (and never below MSM_FAT points)
  uint32_t fat_threshold = (uint32_t)(4 * (n >> (p.c - 1)));  // 4 x the mean bucket size
  if (fat_threshold < fat_min) fat_threshold = fat_min;
  k_msm_scan<<<(unsigned)nw, 256, 0, st>>>(counts, offsets, cursor, p.B, n, fat_counters, fat_items, fat_buckets, max_items,
                                   fat_threshold);
  LAUNCHED(ctx);
  (seg ? k_msm_scatter<true> : k_msm_scatter<false>)<<<(unsigned)((N + 127) / 128), 128, 0, st>>>((const Fr*)canon, N, cursor,
                                                                                                  (uint32_t*)idx, p.c, p.nw, n);
  LAUNCHED(ctx);
  // buckets by decreasing size; empty ones stay the identity (all-zero Jacobian: Z = 0)
  void* ordbuf;
  OK(scratch(ctx, 30, (WB + fat_threshold + 8) * sizeof(uint32_t), &ordbuf));
  uint32_t* size_hist = (uint32_t*)ordbuf;            // fat_threshold + 1 bins; [0] = number of sorted buckets
  uint32_t* order = size_hist + fat_threshold + 8;
  CU(cudaMemsetAsync(size_hist, 0, (fat_threshold + 1) * sizeof(uint32_t), st));
  CU(cudaMemsetAsync(bkt, 0, WB * sizeof(Jac<F>), st));
  k_msm_size_hist<<<(unsigned)((WB + 255) / 256), 256, 0, st>>>(counts, WB, fat_threshold, size_hist);
  LAUNCHED(ctx);
  k_msm_size_scan<<<1, 32, 0, st>>>(size_hist, fat_threshold);
  LAUNCHED(ctx);
  // the scan leaves the start of each size class in its bin: the scatter advances them, bin 0 keeps the total
  k_msm_size_scatter<<<(unsigned)((WB + 255) / 256), 256, 0, st>>>(counts, WB, fat_threshold, size_hist, order);
  LAUNCHED(ctx);
  ts_.reset();
  ts_.emplace(ctx, RIPP_T_MSM);
  (seg ? k_msm_accumulate<F, true> : k_msm_accumulate<F, false>)<<<(unsigned)((WB + 127) / 128), 128, 0, st>>>(bases, (const uint32_t*)idx, offsets, counts,
                                                                   (Jac<F>*)bkt, order, size_hist, (uint32_t)seg_buckets,
                                                                   bases_stride);
  LAUNCHED(ctx);
  {
    unsigned fat_grid = max_items < 1184u ? max_items : 1184u;  // grid-stride over the item list; 8 blocks per SM
    (seg ? k_msm_fat_chunks<F, true> : k_msm_fat_chunks<F, false>)<<<fat_grid, 128, 0, st>>>(bases, (const uint32_t*)idx, offsets, counts, fat_counters, fat_items,
                                                  fat_partials, (uint32_t)seg_buckets, bases_stride);
    LAUNCHED(ctx);
    k_msm_fat_combine<F><<<max_fat < 256u ? max_fat : 256u, 64, 0, st>>>(fat_counters, fat_buckets, fat_partials, (Jac<F>*)bkt);
    LAUNCHED(ctx);
  }
  ts_.reset();
  ts_.emplace(ctx, RIPP_T_MSM_REDUCE);
  size_t WT = nw * p.T;
  Jac<F>* pa = (Jac<F>*)parts;
  Jac<F>* pb = pa + WT;
  k_msm_bucket_reduce<F><<<(unsigned)((WT + 127) / 128), 128, 0, st>>>((const Jac<F>*)bkt, p.B, p.L, p.T, pa, WT);
  LAUNCHED(ctx);
  // window sums: one block per window (strided partial sums, then a shared-memory tree) instead of a ladder of
  // log_8(T) launches of a few warps each
  k_msm_window_sum<F><<<(unsigned)nw, WSUM_THREADS<F>::N, 0, st>>>(pa, p.T, pb);
  LAUNCHED(ctx);
  pa = pb;
  if (fold_mode() == 0) {
    typedef xt::TeamOf<F> TO;
    int warps = (p.nw + TO::PER_WARP - 1) / TO::PER_WARP;
    if (warps > 9) warps = 9;
    k_msm_horner_xt<F><<<(unsigned)nseg, 32 * warps, horner_xt_smem<F>(p.nw), st>>>(pa, p.nw, p.c, out);
  } else if (fold_mode() == 1) {
    typedef typename X3Of<F>::type XF;
    k_msm_horner_x3<XF><<<(unsigned)nseg, 96, 0, st>>>((const Jac<XF>*)pa, p.nw, p.c, (Aff<XF>*)out);
  } else {
    k_msm_horner<F><<<(unsigned)nseg, 32, 0, st>>>(pa, p.nw, p.c, out);
  }
  LAUNCHED(ctx);
  return RIPP_OK;
}

extern "C" int ripp_msm_g1_dev(ripp_ctx* ctx, const void* bases, const void* sc, size_t n, void* out) {
  if (!ctx || !out || (n && (!bases || !sc))) return fail(RIPP_ERR_ARG, "null argument");
  return msm_dev<Fq>(ctx, (const G1Aff*)bases, (const Fr*)sc, n, (G1Aff*)out);
}
extern "C" int ripp_msm_g2_dev(ripp_ctx* ctx, const void* bases, const void* sc, size_t n, void* out) {
  if (!ctx || !out || (n && (!bases || !sc))) return fail(RIPP_ERR_ARG, "null argument");
  return msm_dev<Fq2>(ctx, (const G2Aff*)bases, (const Fr*)sc, n, (G2Aff*)out);
}

// nseg MSMs in one pass (segmented Pippenger above); the scalars of segment s at sc + s sc_stride
int ripp_msm_batch_internal(ripp_ctx* ctx, int group, const void* bases, size_t bases_stride, const void* sc, size_t sc_stride,
                            size_t n, size_t nseg, void* out) {
  if (nseg == 0) return RIPP_OK;
  if (group == 1) return msm_dev<Fq>(ctx, (const G1Aff*)bases, (const Fr*)sc, n, (G1Aff*)out, nseg, bases_stride, sc_stride);
  return msm_dev<Fq2>(ctx, (const G2Aff*)bases, (const Fr*)sc, n, (G2Aff*)out, nseg, bases_stride, sc_stride);
}
static int msm_batch_entry(ripp_ctx* ctx, int group, const void* bases, size_t bases_stride, const void* sc, size_t n, size_t nseg,
                           void* out) {
  if (!ctx || (nseg && !out) || (n && nseg && (!bases || !sc))) return fail(RIPP_ERR_ARG, "null argument");
  // the workspace grows with both: ~65 KB per short G2 segment (window by segment length), and for long ones that of
  // one MSM over all nseg x n points
  if (nseg > ((size_t)1 << 16)) return fail(RIPP_ERR_ARG, "batch MSM: more than 2^16 segments");
  if (n && nseg > ((size_t)1 << 24) / n) return fail(RIPP_ERR_ARG, "batch MSM: segments x length over 2^24");
  return ripp_msm_batch_internal(ctx, group, bases, bases_stride, sc, n, n, nseg, out);
}
extern "C" int ripp_msm_g1_batch_dev(ripp_ctx* ctx, const void* bases, size_t bases_stride, const void* sc, size_t n, size_t nseg,
                                     void* out) {
  return msm_batch_entry(ctx, 1, bases, bases_stride, sc, n, nseg, out);
}
extern "C" int ripp_msm_g2_batch_dev(ripp_ctx* ctx, const void* bases, size_t bases_stride, const void* sc, size_t n, size_t nseg,
                                     void* out) {
  return msm_batch_entry(ctx, 2, bases, bases_stride, sc, n, nseg, out);
}

template <class F>
__global__ void k_normalize_any(const Jac<F>* __restrict__ in, Aff<F>* __restrict__ out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Jac<F> p = in[i];
  out[i] = p.is_inf() ? Aff<F>::inf() : (p.z == F::one() ? Aff<F>{p.x, p.y} : p.to_affine());
}
template <class F>
__global__ void k_aff_to_jac(const Aff<F>* __restrict__ in, Jac<F>* __restrict__ out, size_t n) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = Jac<F>::from_affine(in[i]);
}

// MultiexponentiationInnerProduct::inner_product (inner_products/src/lib.rs:123-142), host pointers
template <class F>
static int msm_host(ripp_ctx* ctx, const void* bases_jac, size_t nl, const void* sc, size_t nr, void* out_jac) {
  if (!ctx || !out_jac) return fail(RIPP_ERR_ARG, "null argument");
  if (nl != nr)
    return fail(RIPP_ERR_LEN_MISMATCH, "left length, right length: " + std::to_string(nl) + ", " + std::to_string(nr));
  size_t n = nl;
  if (n && (!bases_jac || !sc)) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  size_t o_sc = (n * sizeof(Jac<F>) + 255) & ~(size_t)255;
  size_t o_aff = o_sc + ((n * sizeof(Fr) + 255) & ~(size_t)255);
  size_t o_out = o_aff + ((n * sizeof(Aff<F>) + 255) & ~(size_t)255);
  void* buf;
  OK(scratch(ctx, 0, o_out + 1024, &buf));
  char* d = (char*)buf;
  if (n) {
    CU(cudaMemcpyAsync(d, bases_jac, n * sizeof(Jac<F>), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d + o_sc, sc, n * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
    k_normalize_any<F><<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>((const Jac<F>*)d, (Aff<F>*)(d + o_aff), n);
    LAUNCHED(ctx);
  }
  OK(msm_dev<F>(ctx, (const Aff<F>*)(d + o_aff), (const Fr*)(d + o_sc), n, (Aff<F>*)(d + o_out)));
  k_aff_to_jac<F><<<1, 32, 0, ctx->stream>>>((const Aff<F>*)(d + o_out), (Jac<F>*)(d + o_out + 512), 1);
  LAUNCHED(ctx);
  CU(cudaMemcpyAsync(out_jac, d + o_out + 512, sizeof(Jac<F>), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}
extern "C" int ripp_msm_g1(ripp_ctx* ctx, const void* b, size_t nl, const void* s, size_t nr, void* out) {
  return msm_host<Fq>(ctx, b, nl, s, nr, out);
}
extern "C" int ripp_msm_g2(ripp_ctx* ctx, const void* b, size_t nl, const void* s, size_t nr, void* out) {
  return msm_host<Fq2>(ctx, b, nl, s, nr, out);
}

// ------------------------------------------------------------------------------------------------
// folds with one scalar shared by all elements: out[i] = hi[i] * c + lo[i]
// ------------------------------------------------------------------------------------------------
// The scalar shared by a whole fold is recoded once on the host into non-adjacent form: digit i is
// +1 / -1 / 0 according to bit i of `pos` / `neg`.  NAF has ~n/3 non-zero digits instead of ~n/2, i.e. a third
// fewer additions on every element's (latency-bound) double-and-add chain; c = sum digit_i 2^i exactly.
struct ScalarBits {
  uint32_t pos[9], neg[9];
  int nbits;  // digits
};

static ScalarBits scalar_bits(const void* fr_mont_host) {
  Fr s;
  memcpy(s.v, fr_mont_host, sizeof(Fr));
  s = s.from_mont();
  uint32_t k[10] = {0};
  for (int i = 0; i < 8; i++) k[i] = s.v[i];
  ScalarBits b;
  memset(&b, 0, sizeof(b));
  int i = 0;
  auto is_zero = [&] { for (int j = 0; j < 10; j++) if (k[j]) return false; return true; };
  while (!is_zero()) {
    if (k[0] & 1) {
      int d = 2 - (int)(k[0] & 3);  // +1 if k = 1 mod 4, -1 if k = 3 mod 4
      if (d == 1) {
        b.pos[i >> 5] |= 1u << (i & 31);
        k[0] -= 1;
      } else {
        b.neg[i >> 5] |= 1u << (i & 31);
        for (int j = 0; j < 10; j++) {  // k += 1
          if (++k[j]) break;
        }
      }
    }
    for (int j = 0; j < 9; j++) k[j] = (k[j] >> 1) | (k[j + 1] << 31);
    k[9] >>= 1;
    i++;
  }
  b.nbits = i;
  return b;
}

// ---- endomorphism-accelerated folds -----------------------------------------------------------------
// The shared scalar is split on the host into m short digits in base B (G1: B = lambda = x^2 - 1, two 128-bit
// digits; G2: B = |x|, up to four 64-bit digits), c = sum_i d_i B^i, and  c P = sum_i d_i E^i(P)  with the
// cheap map E = phi (G1) / -psi (G2): a joint double-and-add over max|d_i| bits instead of |c| bits.
template <class F>
static EndoBits endo_bits(const void* fr_mont_host) {
  Fr s;
  memcpy(s.v, fr_mont_host, sizeof(Fr));
  s = s.from_mont();
  EndoBits b;
  endo_decompose<sizeof(F) == sizeof(Fq) ? 1 : 2>(s.v, b);
  return b;
}

template <class F>
__global__ void __launch_bounds__(64, 4) k_fold_endo(const Aff<F>* __restrict__ hi, const Aff<F>* __restrict__ lo, EndoBits c,
                                                     size_t n, Aff<F>* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Jac<F> acc = endo_mul<F>(hi[i], c);
  acc = acc.add_mixed(lo[i]);
  out[i] = acc.to_affine();
}

template <class F>
__global__ void __launch_bounds__(64, 4) k_fold(const Aff<F>* __restrict__ hi, const Aff<F>* __restrict__ lo, ScalarBits c,
                                                size_t n, Aff<F>* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  Aff<F> p = hi[i], np = p.neg();
  Jac<F> acc = Jac<F>::inf();
  for (int j = c.nbits - 1; j >= 0; j--) {
    acc = acc.dbl();
    if ((c.pos[j >> 5] >> (j & 31)) & 1) acc = acc.add_mixed(p);
    if ((c.neg[j >> 5] >> (j & 31)) & 1) acc = acc.add_mixed(np);
  }
  acc = acc.add_mixed(lo[i]);
  out[i] = acc.to_affine();
}

// one three-warp team per 32 elements (x3.cuh): XF = Fq for G1, x3::Fq2x3 for G2 (same memory layout as Fq / Fq2).
// Every thread stays to the end (the exchanges are CTA barriers): lanes past n work on element n - 1 and do not store.
template <class XF>
__global__ void __maxnreg__(255) k_fold_w3(const Aff<XF>* __restrict__ hi, const Aff<XF>* __restrict__ lo, EndoBits c,
                                                size_t n, Aff<XF>* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * 32 + (threadIdx.x & 31);
  const bool live = i < n;
  if (!live) i = n - 1;
  Jac<XF> acc = x3::endo_mul<XF>(hi[i], c);
  acc = x3::Ops<XF>::madd(acc, lo[i]);
  Aff<XF> o = x3::to_affine(acc);
  if (live && threadIdx.x < 32) out[i] = o;
}

// lane teams (xt.cuh): 3 lanes per G1 element (10 per warp), 9 lanes per G2 element (3 per warp); the remaining lanes
// mirror the first ones (same element, same bus slice: identical values), elements past n redo element n - 1 on their
// own bus slice and do not store.
constexpr int XT_WARPS = 2;
template <class F>
__global__ void __launch_bounds__(32 * XT_WARPS) k_fold_xt(const Aff<F>* __restrict__ hi, const Aff<F>* __restrict__ lo, EndoBits c,
                                                           size_t n, Aff<F>* __restrict__ out) {
  typedef xt::TeamOf<F> TO;
  constexpr int AW4 = 4 * sizeof(Aff<F>) / 4;  // four endomorphism images of the element
  __shared__ __align__(16) uint32_t bus[XT_WARPS * TO::PER_WARP * (2 * TO::BUS_WORDS + AW4)];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int vl = lane % (TO::LANES * TO::PER_WARP);
  const int e = vl / TO::LANES;
  size_t i = ((size_t)blockIdx.x * XT_WARPS + warp) * TO::PER_WARP + e;
  const bool live = i < n && lane == vl;
  if (i >= n) i = n - 1;
  uint32_t* scratch = bus + (warp * TO::PER_WARP + e) * (2 * TO::BUS_WORDS + AW4);
  xt::Team tm{vl % TO::LANES, scratch, 0, nullptr};
  Jac<F> acc = xt::endo_mul<F>(tm, hi[i], c, scratch + 2 * TO::BUS_WORDS);
  acc = xt::madd<F>(tm, acc, lo[i]);
  Aff<F> o = xt::to_affine<F>(tm, acc);
  if (live && tm.t == 0) out[i] = o;
}
// vectors up to this length run on lane teams (RIPP_B200_XT_MAX overrides).  Re-measured at the end of round 2 on the 2^12
// aggregation (profiles/r2zi_last_call_xt_max.json): 67.2 ms at 2048, 64.8 at 1024, 65.8 at 512, 65.2 at 256 -- the four
// 2048-element folds of the first round (1776 warps of teams in one launch, 3.7 ms) are served better by one thread per
// element on four streams; from 1024 elements down the teams win.
static size_t xt_max_n() {
  static const long v = [] {
    const char* e = getenv("RIPP_B200_XT_MAX");
    return e ? atol(e) : 1024L;
  }();
  return (size_t)v;
}

// ---- the folds of ONE GIPA round in ONE launch (gipa.rs:261-291: A, B, v, w rescaled together) ------------------
// Up to four jobs (G1 / G2 on lane teams, Fr one thread per element); blocks [first_block, first_block + blocks) of the
// grid belong to a job, so a block runs exactly one of the three bodies.  Same arithmetic as k_fold_xt / k_fr_fold.
struct FoldJob {
  int type;  // 0 = none, 1 = G1, 2 = G2, 3 = Fr
  const void* hi;
  const void* lo;
  void* out;
  uint32_t n, first_block;
  EndoBits c;  // G1 / G2
  Fr s;        // Fr
  // fold with precomputed bases (k_fold4_xp<true>): D_i = [2^H] hi_i written by k_fold_pre, and c split at bit H
  const void* pre;
  EndoSplit cs;
};
struct FoldJobs {
  FoldJob j[4];
};
template <class F>
__device__ __forceinline__ void fold_xt_body(uint32_t* bus, const FoldJob& job, uint32_t block) {
  typedef xt::TeamOf<F> TO;
  constexpr int AW4 = 4 * sizeof(Aff<F>) / 4;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int vl = lane % (TO::LANES * TO::PER_WARP);
  const int e = vl / TO::LANES;
  size_t i = ((size_t)block * XT_WARPS + warp) * TO::PER_WARP + e;
  const bool live = i < job.n && lane == vl;
  if (i >= job.n) i = job.n - 1;
  uint32_t* scratch = bus + (warp * TO::PER_WARP + e) * (2 * TO::BUS_WORDS + AW4);
  xt::Team tm{vl % TO::LANES, scratch, 0, nullptr};
  Jac<F> acc = xt::endo_mul<F>(tm, ((const Aff<F>*)job.hi)[i], job.c, scratch + 2 * TO::BUS_WORDS);
  acc = xt::madd<F>(tm, acc, ((const Aff<F>*)job.lo)[i]);
  Aff<F> o = xt::to_affine<F>(tm, acc);
  if (live && tm.t == 0) ((Aff<F>*)job.out)[i] = o;
}
constexpr int FOLD4_BUS_WORDS_G1 = XT_WARPS * xt::TeamOf<Fq>::PER_WARP * (2 * xt::TeamOf<Fq>::BUS_WORDS + 4 * 24);
constexpr int FOLD4_BUS_WORDS_G2 = XT_WARPS * xt::TeamOf<Fq2>::PER_WARP * (2 * xt::TeamOf<Fq2>::BUS_WORDS + 4 * 48);
__global__ void __launch_bounds__(32 * XT_WARPS) k_fold4_xt(const FoldJobs jobs) {
  __shared__ __align__(16) uint32_t bus[FOLD4_BUS_WORDS_G1 > FOLD4_BUS_WORDS_G2 ? FOLD4_BUS_WORDS_G1 : FOLD4_BUS_WORDS_G2];
  int k = 0;
#pragma unroll
  for (int t = 1; t < 4; t++)
    if (jobs.j[t].type && blockIdx.x >= jobs.j[t].first_block) k = t;
  const FoldJob& job = jobs.j[k];
  const uint32_t block = blockIdx.x - job.first_block;
  if (job.type == 1) {
    fold_xt_body<Fq>(bus, job, block);
  } else if (job.type == 2) {
    fold_xt_body<Fq2>(bus, job, block);
  } else if (job.type == 3) {
    size_t i = (size_t)block * blockDim.x + threadIdx.x;
    if (i < job.n) ((Fr*)job.out)[i] = ((const Fr*)job.hi)[i] * job.s + ((const Fr*)job.lo)[i];
  }
}
// Part-parallel variant for the short vectors of the late rounds (n <= xp_max_n()): a CTA of four warps; warp w works
// on endomorphism part w % m of the elements of group w / m (m = 4 parts for G2: one group of 3 elements per CTA; m = 2
// for G1: two groups of 10), every team brings its part to affine form, and after the CTA barrier the part-0 warp adds
// lo and the m parts.  Same group element as fold_xt_body (the sum is exact), half the dependent chain.
// PRE: the split recoding (endo.cuh: endo_split) over the bases {E^k(hi_i), E^k(D_i)}, D_i = job.pre[i] = [2^H] hi_i
// precomputed by k_fold_pre while the round's products ran: twice the parts (G1 4, G2 8) at half the chain, eight warps.
template <bool PRE>
struct XpShape {
  static constexpr int WARPS = PRE ? 8 : 4;
  template <class F>  // the layout does not depend on the scalar: the group's full part count
  static constexpr int PARTS = (sizeof(F) == sizeof(Fq) ? 2 : 4) * (PRE ? 2 : 1);
};
constexpr int XP_WARPS = XpShape<false>::WARPS;
template <class F, int WARPS>
struct XpLayout {
  typedef xt::TeamOf<F> TO;
  static constexpr int AW = sizeof(Aff<F>) / 4;
  static constexpr int TEAM_WORDS = 2 * TO::BUS_WORDS + AW;
  static constexpr int PARTS_AT = WARPS * TO::PER_WARP * TEAM_WORDS;
  static constexpr int WORDS = PARTS_AT + WARPS * TO::PER_WARP * AW;  // (group, element, part) slots: groups * m = WARPS
};
template <class F, bool PRE>
__device__ __forceinline__ void fold_xp_body(uint32_t* sm, const FoldJob& job, uint32_t block) {
  typedef xt::TeamOf<F> TO;
  constexpr int WARPS = XpShape<PRE>::WARPS;
  typedef XpLayout<F, WARPS> L;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  constexpr int m = XpShape<PRE>::template PARTS<F>;
  constexpr int mk = PRE ? m / 2 : m;  // powers of E
  const int part = warp % m, grp = warp / m, groups = WARPS / m;
  const int vl = lane % (TO::LANES * TO::PER_WARP);
  const int e = vl / TO::LANES;
  size_t i = ((size_t)block * groups + grp) * TO::PER_WARP + e;
  const bool live = i < job.n && lane == vl;
  if (i >= job.n) i = job.n - 1;
  uint32_t* scratch = sm + (warp * TO::PER_WARP + e) * L::TEAM_WORDS;
  uint32_t* slots = sm + L::PARTS_AT + ((grp * TO::PER_WARP + e) * m) * L::AW;
  xt::Team tm{vl % TO::LANES, scratch, 0, nullptr};
  {
    Jac<F> acc;
    if (PRE) {
      const Aff<F>* src = (const Aff<F>*)((part & 1) ? job.pre : job.hi);
      acc = xt::naf_mul_endo<F>(tm, src[i], mk, part >> 1, job.cs.pos[part], job.cs.neg[part], job.cs.nbits[part],
                                scratch + 2 * TO::BUS_WORDS);
    } else {
      acc = xt::part_mul<F>(tm, ((const Aff<F>*)job.hi)[i], job.c, mk, part, scratch + 2 * TO::BUS_WORDS);
    }
    Aff<F> pa = xt::to_affine<F>(tm, acc);
    if (tm.t == 0 && lane == vl) xt::aff_st<F>(slots + part * L::AW, pa);
  }
  __syncthreads();
  if (part == 0) {
    Jac<F> s = Jac<F>::from_affine(((const Aff<F>*)job.lo)[i]);
#pragma unroll 1
    for (int t = 0; t < m; t++) s = xt::madd<F>(tm, s, xt::aff_ld<F>(slots + t * L::AW));
    Aff<F> o = xt::to_affine<F>(tm, s);
    if (live && tm.t == 0) ((Aff<F>*)job.out)[i] = o;
  }
}
template <bool PRE>
__global__ void __launch_bounds__(32 * XpShape<PRE>::WARPS) k_fold4_xp(const FoldJobs jobs) {
  constexpr int W1 = XpLayout<Fq, XpShape<PRE>::WARPS>::WORDS, W2 = XpLayout<Fq2, XpShape<PRE>::WARPS>::WORDS;
  __shared__ __align__(16) uint32_t sm[W1 > W2 ? W1 : W2];
  int k = 0;
#pragma unroll
  for (int t = 1; t < 4; t++)
    if (jobs.j[t].type && blockIdx.x >= jobs.j[t].first_block) k = t;
  const FoldJob& job = jobs.j[k];
  const uint32_t block = blockIdx.x - job.first_block;
  if (job.type == 1) {
    fold_xp_body<Fq, PRE>(sm, job, block);
  } else if (job.type == 2) {
    fold_xp_body<Fq2, PRE>(sm, job, block);
  } else if (job.type == 3) {
    size_t i = (size_t)block * blockDim.x + threadIdx.x;
    if (i < job.n) ((Fr*)job.out)[i] = ((const Fr*)job.hi)[i] * job.s + ((const Fr*)job.lo)[i];
  }
}

// D_i = [2^H] hi_i for the G1 / G2 jobs of a round (job.out = the fold's `pre`): lane teams as k_fold4_xt, no scalar.
// Runs on its own stream while the round's products and its challenge are computed.
__global__ void __launch_bounds__(32 * XT_WARPS) k_fold_pre(const FoldJobs jobs) {
  constexpr int W1 = xt::TeamOf<Fq>::PER_WARP * 2 * xt::TeamOf<Fq>::BUS_WORDS;
  constexpr int W2 = xt::TeamOf<Fq2>::PER_WARP * 2 * xt::TeamOf<Fq2>::BUS_WORDS;
  __shared__ __align__(16) uint32_t bus[XT_WARPS * (W1 > W2 ? W1 : W2)];
  int k = 0;
#pragma unroll
  for (int t = 1; t < 4; t++)
    if (jobs.j[t].type && blockIdx.x >= jobs.j[t].first_block) k = t;
  const FoldJob& job = jobs.j[k];
  const uint32_t block = blockIdx.x - job.first_block;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (job.type == 1) {
    typedef xt::TeamOf<Fq> TO;
    const int vl = lane % (TO::LANES * TO::PER_WARP), e = vl / TO::LANES;
    size_t i = ((size_t)block * XT_WARPS + warp) * TO::PER_WARP + e;
    const bool live = i < job.n && lane == vl;
    if (i >= job.n) i = job.n - 1;
    xt::Team tm{vl % TO::LANES, bus + (warp * TO::PER_WARP + e) * 2 * TO::BUS_WORDS, 0, nullptr};
    G1Aff d = xt::pow2_mul<Fq>(tm, ((const G1Aff*)job.hi)[i], SplitOf<1>::H);
    if (live && tm.t == 0) ((G1Aff*)job.out)[i] = d;
  } else if (job.type == 2) {
    typedef xt::TeamOf<Fq2> TO;
    const int vl = lane % (TO::LANES * TO::PER_WARP), e = vl / TO::LANES;
    size_t i = ((size_t)block * XT_WARPS + warp) * TO::PER_WARP + e;
    const bool live = i < job.n && lane == vl;
    if (i >= job.n) i = job.n - 1;
    xt::Team tm{vl % TO::LANES, bus + (warp * TO::PER_WARP + e) * 2 * TO::BUS_WORDS, 0, nullptr};
    G2Aff d = xt::pow2_mul<Fq2>(tm, ((const G2Aff*)job.hi)[i], SplitOf<2>::H);
    if (live && tm.t == 0) ((G2Aff*)job.out)[i] = d;
  }
}
// vectors up to this length fold part-parallel (RIPP_B200_XP_MAX overrides; 0 = never).  Measured on the 2^12 aggregation
// (gpurun_out r2i): launch 1.25 ms against 1.45-1.6 ms for k_fold4_xt at n <= 128 (the G1 vectors' 128-bit parts are
// the chain that remains), level at n = 256, slower above; whole aggregation 72.6 / 73.9 / 75.3 ms at 128 / 256 / 512.
static size_t xp_max_n() {
  static const long v = [] {
    const char* e = getenv("RIPP_B200_XP_MAX");
    return e ? atol(e) : 128L;
  }();
  return (size_t)v;
}

// vectors up to this length fold with precomputed bases (RIPP_B200_FOLD_PRE_MAX overrides; 0 = never); never above
// the lane-team range, and not under a forced fold kernel.  Measured on the 2^12 aggregation (profiles/r3a_fold_pre.json):
// 62.8 ms at 128 against 64.9 with none, 63.1 at 256, 70.1 at 1024 (there the precompute competes with the Miller kernels).
size_t ripp_fold_pre_max_n() {
  static const long v = [] {
    const char* e = getenv("RIPP_B200_FOLD_PRE_MAX");
    return e ? atol(e) : 128L;
  }();
  if (fold_mode() != 0 || v <= 0) return 0;
  return (size_t)v < xt_max_n() ? (size_t)v : xt_max_n();
}

// pre[t] = [2^H] hi[t] (n elements each) for the G1 / G2 entries of types[] (others ignored), on ctx's stream
int ripp_fold_pre_internal(ripp_ctx* ctx, const int* types, const void* const* hi, size_t n, void* const* pre) {
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  FoldJobs jobs;
  memset(&jobs, 0, sizeof(jobs));
  uint32_t nblocks = 0;
  int nj = 0;
  for (int t = 0; t < 4; t++) {
    if ((types[t] != 1 && types[t] != 2) || !hi[t]) continue;
    FoldJob& j = jobs.j[nj++];
    j.type = types[t];
    j.hi = hi[t];
    j.out = pre[t];
    j.n = (uint32_t)n;
    j.first_block = nblocks;
    const uint32_t per = types[t] == 1 ? xt::TeamOf<Fq>::PER_WARP : xt::TeamOf<Fq2>::PER_WARP;
    const uint32_t warps = (uint32_t)((n + per - 1) / per);
    nblocks += (warps + XT_WARPS - 1) / XT_WARPS;
  }
  if (!nj) return RIPP_OK;
  TimeScope ts_(ctx, RIPP_T_FOLD);
  k_fold_pre<<<nblocks, 32 * XT_WARPS, 0, ctx->stream>>>(jobs);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// types[t] in {0 none, 1 G1, 2 G2, 3 Fr}; out[t][i] = hi[t][i] * c[t] + lo[t][i].  Returns RIPP_OK and *fused = 1 when the
// fused launch was used (all vectors short enough for lane teams), *fused = 0 when the caller should fold one by one.
// pre: NULL, or per job the [2^H] hi images that ripp_fold_pre_internal wrote (then the G1 / G2 folds run
// k_fold4_xp<true>, whatever the part-parallel range)
int ripp_fold4_internal(ripp_ctx* ctx, const int* types, const void* const* hi, const void* const* lo, const void* const* cs, size_t n,
                        void* const* out, int* fused, const void* const* pre) {
  *fused = 0;
  if (fold_mode() != 0 || n == 0 || n > xt_max_n()) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  FoldJobs jobs;
  memset(&jobs, 0, sizeof(jobs));
  uint32_t nblocks = 0;
  int nj = 0;
  const bool xp = pre || n <= xp_max_n();
  const int xp_warps = pre ? XpShape<true>::WARPS : XP_WARPS;
  for (int t = 0; t < 4; t++) {
    if (!types[t] || !hi[t]) continue;
    FoldJob& j = jobs.j[nj++];
    j.type = types[t];
    j.hi = hi[t];
    j.lo = lo[t];
    j.out = out[t];
    j.n = (uint32_t)n;
    j.first_block = nblocks;
    uint32_t blocks;
    if (types[t] == 1) {
      j.c = endo_bits<Fq>(cs[t]);
      if (pre) {
        j.pre = pre[t];
        endo_split<1>(j.c, j.cs);
      }
      uint32_t warps = (uint32_t)((n + xt::TeamOf<Fq>::PER_WARP - 1) / xt::TeamOf<Fq>::PER_WARP);
      const int m = pre ? XpShape<true>::PARTS<Fq> : XpShape<false>::PARTS<Fq>;
      blocks = xp ? (warps * m + xp_warps - 1) / xp_warps : (warps + XT_WARPS - 1) / XT_WARPS;
    } else if (types[t] == 2) {
      j.c = endo_bits<Fq2>(cs[t]);
      if (pre) {
        j.pre = pre[t];
        endo_split<2>(j.c, j.cs);
      }
      uint32_t warps = (uint32_t)((n + xt::TeamOf<Fq2>::PER_WARP - 1) / xt::TeamOf<Fq2>::PER_WARP);
      const int m = pre ? XpShape<true>::PARTS<Fq2> : XpShape<false>::PARTS<Fq2>;
      blocks = xp ? (warps * m + xp_warps - 1) / xp_warps : (warps + XT_WARPS - 1) / XT_WARPS;
    } else {
      memcpy(j.s.v, cs[t], sizeof(Fr));
      const uint32_t bt = 32 * (xp ? xp_warps : XT_WARPS);
      blocks = (uint32_t)((n + bt - 1) / bt);
    }
    nblocks += blocks;
  }
  if (!nj) {
    *fused = 1;
    return RIPP_OK;
  }
  // jobs are packed at the front of the array in launch order: unused slots keep type 0
  TimeScope ts_(ctx, RIPP_T_FOLD);
  if (pre)
    k_fold4_xp<true><<<nblocks, 32 * xp_warps, 0, ctx->stream>>>(jobs);
  else if (xp)
    k_fold4_xp<false><<<nblocks, 32 * xp_warps, 0, ctx->stream>>>(jobs);
  else
    k_fold4_xt<<<nblocks, 32 * XT_WARPS, 0, ctx->stream>>>(jobs);
  LAUNCHED(ctx);
  *fused = 1;
  return RIPP_OK;
}

// ---- the folds of many GIPA recursions from a device table (the lock-step batch prover, aggregate_batch.cuh) ------------
// Sections by element type (G1, G2, Fr); within a section, group g of K jobs folds the vector at base[g] + k stride[g]
// (instance k) with the scalar record sc[g][k] (EndoBits for G1 / G2, Fr for Fr).  All jobs have the same length n, so a
// block finds its job from its section's first block and the blocks per job; the job itself is built in registers and
// handed to the bodies of k_fold4_xt / k_fold4_xp.
__device__ __forceinline__ bool fold_tab_job(const FoldTable& t, uint32_t blk, int type, FoldJob& job, uint32_t* block) {
  const int s = type - 1;
  if (blk < t.first_block[s] || blk >= t.first_block[s] + t.blocks[s]) return false;
  const uint32_t r = blk - t.first_block[s], j = r / t.bpj[s], g = j / t.K, k = j % t.K;
  const size_t esz = type == 1 ? sizeof(G1Aff) : type == 2 ? sizeof(G2Aff) : sizeof(Fr);
  char* lo = t.base[s][g] + (size_t)k * t.stride[s][g];
  job.type = type;
  job.lo = lo;
  job.hi = lo + (size_t)t.n * esz;
  job.out = lo;
  job.n = t.n;
  if (type == 3)
    job.s = ((const Fr*)t.sc[s][g])[k];
  else
    job.c = ((const EndoBits*)t.sc[s][g])[k];
  *block = r - j * t.bpj[s];
  return true;
}
template <bool XP>
__global__ void __launch_bounds__(32 * (XP ? XP_WARPS : XT_WARPS)) k_fold_tab(const FoldTable t) {
  constexpr int W1 = XP ? XpLayout<Fq, XP_WARPS>::WORDS : FOLD4_BUS_WORDS_G1;
  constexpr int W2 = XP ? XpLayout<Fq2, XP_WARPS>::WORDS : FOLD4_BUS_WORDS_G2;
  __shared__ __align__(16) uint32_t sm[W1 > W2 ? W1 : W2];
  FoldJob job;
  uint32_t block;
  if (fold_tab_job(t, blockIdx.x, 1, job, &block)) {
    if constexpr (XP) fold_xp_body<Fq, false>(sm, job, block);
    else fold_xt_body<Fq>(sm, job, block);
  } else if (fold_tab_job(t, blockIdx.x, 2, job, &block)) {
    if constexpr (XP) fold_xp_body<Fq2, false>(sm, job, block);
    else fold_xt_body<Fq2>(sm, job, block);
  } else if (fold_tab_job(t, blockIdx.x, 3, job, &block)) {
    size_t i = (size_t)block * blockDim.x + threadIdx.x;
    if (i < job.n) ((Fr*)job.out)[i] = ((const Fr*)job.hi)[i] * job.s + ((const Fr*)job.lo)[i];
  }
}
// long vectors (above the lane-team range): one thread per element, one launch per element type; the table holds only
// that type's section at first block 0
template <class F>
__global__ void __launch_bounds__(64, 4) k_fold_tab_endo(const FoldTable t) {
  constexpr int type = sizeof(F) == sizeof(Fq) ? 1 : 2;
  FoldJob job;
  uint32_t block;
  if (!fold_tab_job(t, blockIdx.x, type, job, &block)) return;
  size_t i = (size_t)block * blockDim.x + threadIdx.x;
  if (i >= job.n) return;
  Jac<F> acc = endo_mul<F>(((const Aff<F>*)job.hi)[i], job.c);
  acc = acc.add_mixed(((const Aff<F>*)job.lo)[i]);
  ((Aff<F>*)job.out)[i] = acc.to_affine();
}
__global__ void k_fold_tab_fr(const FoldTable t) {
  FoldJob job;
  uint32_t block;
  if (!fold_tab_job(t, blockIdx.x, 3, job, &block)) return;
  size_t i = (size_t)block * blockDim.x + threadIdx.x;
  if (i < job.n) ((Fr*)job.out)[i] = ((const Fr*)job.hi)[i] * job.s + ((const Fr*)job.lo)[i];
}

// host side of the scalar records
void ripp_endo_bits(int group, const void* fr_mont_host, EndoBits* out) {
  *out = group == 1 ? endo_bits<Fq>(fr_mont_host) : endo_bits<Fq2>(fr_mont_host);
}

// One round's folds of every job in t (t.base / stride / sc / ngroups / K / n filled by the caller): one launch while
// the vectors are short enough for lane teams, else one launch per element type.  The RIPP_B200_FOLD override of the
// single path (A/B runs of the fold kernels) does not apply here: the batch always runs these kernels, and the result
// does not depend on the kernel.
int ripp_fold_table_internal(ripp_ctx* ctx, FoldTable t) {
  const size_t n = t.n;
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  TimeScope ts_(ctx, RIPP_T_FOLD);
  if (n <= xt_max_n()) {
    const bool xp = n <= xp_max_n();
    const uint32_t bt = 32 * (xp ? XP_WARPS : XT_WARPS);
    uint32_t nblocks = 0;
    for (int s = 0; s < 3; s++) {
      uint32_t bpj;
      if (s < 2) {
        const uint32_t per = s == 0 ? xt::TeamOf<Fq>::PER_WARP : xt::TeamOf<Fq2>::PER_WARP;
        const uint32_t warps = (uint32_t)((n + per - 1) / per);
        const int m = s == 0 ? XpShape<false>::PARTS<Fq> : XpShape<false>::PARTS<Fq2>;
        bpj = xp ? (warps * m + XP_WARPS - 1) / XP_WARPS : (warps + XT_WARPS - 1) / XT_WARPS;
      } else {
        bpj = (uint32_t)((n + bt - 1) / bt);
      }
      t.bpj[s] = bpj;
      t.first_block[s] = nblocks;
      t.blocks[s] = bpj * t.K * t.ngroups[s];
      nblocks += t.blocks[s];
    }
    if (xp)
      k_fold_tab<true><<<nblocks, bt, 0, ctx->stream>>>(t);
    else
      k_fold_tab<false><<<nblocks, bt, 0, ctx->stream>>>(t);
    LAUNCHED(ctx);
    return RIPP_OK;
  }
  for (int s = 0; s < 3; s++) {
    if (!t.ngroups[s]) continue;
    FoldTable u = t;
    const uint32_t bt = s < 2 ? 64 : 128;
    for (int o = 0; o < 3; o++) u.blocks[o] = 0;
    u.bpj[s] = (uint32_t)((n + bt - 1) / bt);
    u.first_block[s] = 0;
    u.blocks[s] = u.bpj[s] * t.K * t.ngroups[s];
    if (s == 0)
      k_fold_tab_endo<Fq><<<u.blocks[s], bt, 0, ctx->stream>>>(u);
    else if (s == 1)
      k_fold_tab_endo<Fq2><<<u.blocks[s], bt, 0, ctx->stream>>>(u);
    else
      k_fold_tab_fr<<<u.blocks[s], bt, 0, ctx->stream>>>(u);
    LAUNCHED(ctx);
  }
  return RIPP_OK;
}

template <class F, class XF>
static int fold_dev(ripp_ctx* ctx, const void* hi, const void* lo, const void* c, size_t n, void* out) {
  if (!ctx || !c || (n && (!hi || !lo || !out))) return fail(RIPP_ERR_ARG, "null argument");
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  TimeScope ts_(ctx, RIPP_T_FOLD);
  const int mode = fold_mode();
  if (mode == 0 && n <= xt_max_n()) {
    typedef xt::TeamOf<F> TO;
    unsigned warps = (unsigned)((n + TO::PER_WARP - 1) / TO::PER_WARP);
    k_fold_xt<F><<<(warps + XT_WARPS - 1) / XT_WARPS, 32 * XT_WARPS, 0, ctx->stream>>>((const Aff<F>*)hi, (const Aff<F>*)lo,
                                                                                     endo_bits<F>(c), n, (Aff<F>*)out);
  } else if (mode == 1 || (mode == 0 && n <= w3_max_n())) {
    k_fold_w3<XF><<<(unsigned)((n + 31) / 32), 96, 0, ctx->stream>>>((const Aff<XF>*)hi, (const Aff<XF>*)lo, endo_bits<F>(c), n,
                                                                   (Aff<XF>*)out);
  } else if (mode != 3) {
    k_fold_endo<F><<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>((const Aff<F>*)hi, (const Aff<F>*)lo, endo_bits<F>(c), n,
                                                                   (Aff<F>*)out);
  } else {
    k_fold<F><<<(unsigned)((n + 63) / 64), 64, 0, ctx->stream>>>((const Aff<F>*)hi, (const Aff<F>*)lo, scalar_bits(c), n,
                                                              (Aff<F>*)out);
  }
  LAUNCHED(ctx);
  return RIPP_OK;
}
extern "C" int ripp_g1_fold_dev(ripp_ctx* ctx, const void* hi, const void* lo, const void* c, size_t n, void* out) {
  return fold_dev<Fq, Fq>(ctx, hi, lo, c, n, out);
}
extern "C" int ripp_g2_fold_dev(ripp_ctx* ctx, const void* hi, const void* lo, const void* c, size_t n, void* out) {
  return fold_dev<Fq2, x3::Fq2x3>(ctx, hi, lo, c, n, out);
}

__global__ void k_fr_fold(const Fr* __restrict__ hi, const Fr* __restrict__ lo, Fr c, size_t n, Fr* __restrict__ out) {
  size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = hi[i] * c + lo[i];
}
extern "C" int ripp_fr_fold_dev(ripp_ctx* ctx, const void* hi, const void* lo, const void* c, size_t n, void* out) {
  if (!ctx || !c || (n && (!hi || !lo || !out))) return fail(RIPP_ERR_ARG, "null argument");
  if (n == 0) return RIPP_OK;
  CU(cudaSetDevice(ctx->device));
  Fr cc;
  memcpy(cc.v, c, sizeof(Fr));
  k_fr_fold<<<(unsigned)((n + 127) / 128), 128, 0, ctx->stream>>>((const Fr*)hi, (const Fr*)lo, cc, n, (Fr*)out);
  LAUNCHED(ctx);
  return RIPP_OK;
}

// ------------------------------------------------------------------------------------------------
// ScalarInnerProduct (inner_products/src/lib.rs:149-166): sum a_i b_i in Fr
// ------------------------------------------------------------------------------------------------
__global__ void k_fr_dot(const Fr* __restrict__ a, const Fr* __restrict__ b, size_t n, uint32_t R, Fr* __restrict__ out) {
  size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  size_t lo = t * R;
  if (lo >= n) return;
  size_t hi = lo + R < n ? lo + R : n;
  Fr acc = Fr::zero();
  for (size_t j = lo; j < hi; j++) acc = acc + (b ? a[j] * b[j] : a[j]);
  out[t] = acc;
}

extern "C" int ripp_scalar_ip_dev(ripp_ctx* ctx, const void* a, const void* b, size_t n, void* out) {
  if (!ctx || !out || (n && (!a || !b))) return fail(RIPP_ERR_ARG, "null argument");
  CU(cudaSetDevice(ctx->device));
  if (n == 0) {
    CU(cudaMemsetAsync(out, 0, sizeof(Fr), ctx->stream));
    return RIPP_OK;
  }
  const uint32_t R = 16;
  size_t m = (n + R - 1) / R;
  void* buf;
  OK(scratch(ctx, 9, 2 * m * sizeof(Fr) + 64, &buf));
  Fr* pa = (Fr*)buf;
  Fr* pb = pa + m;
  k_fr_dot<<<(unsigned)((m + 127) / 128), 128, 0, ctx->stream>>>((const Fr*)a, (const Fr*)b, n, R, m == 1 ? (Fr*)out : pa);
  LAUNCHED(ctx);
  while (m > 1) {
    size_t mo = (m + R - 1) / R;
    k_fr_dot<<<(unsigned)((mo + 127) / 128), 128, 0, ctx->stream>>>(pa, nullptr, m, R, mo == 1 ? (Fr*)out : pb);
    LAUNCHED(ctx);
    Fr* t = pa;
    pa = pb;
    pb = t;
    m = mo;
  }
  return RIPP_OK;
}

extern "C" int ripp_scalar_ip(ripp_ctx* ctx, const void* a, size_t nl, const void* b, size_t nr, void* out) {
  if (!ctx || !out) return fail(RIPP_ERR_ARG, "null argument");
  if (nl != nr)
    return fail(RIPP_ERR_LEN_MISMATCH, "left length, right length: " + std::to_string(nl) + ", " + std::to_string(nr));
  size_t n = nl;
  CU(cudaSetDevice(ctx->device));
  void* buf;
  OK(scratch(ctx, 0, 2 * n * sizeof(Fr) + 256, &buf));
  Fr* d = (Fr*)buf;
  if (n) {
    CU(cudaMemcpyAsync(d, a, n * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaMemcpyAsync(d + n, b, n * sizeof(Fr), cudaMemcpyHostToDevice, ctx->stream));
  }
  OK(ripp_scalar_ip_dev(ctx, d, d + n, n, d + 2 * n));
  CU(cudaMemcpyAsync(out, d + 2 * n, sizeof(Fr), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return RIPP_OK;
}
