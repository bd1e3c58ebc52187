// Host-simulation build of the fold over precomputed bases (TEST INFRASTRUCTURE ONLY): endo.cuh's split recoding and
// xt.cuh's team formulas, each lane a host thread, in the order k_fold_pre and k_fold4_xp<true> run them.
// Built by tests/test_hostsim_fold_pre.py.
#define RIPP_HOSTSIM 1
#include "../../ripp_b200/csrc/xt.cuh"
#include <pthread.h>
#include <string.h>
#include <thread>
#include <vector>
using namespace ripp;

namespace ripp { namespace xt {
void host_barrier(void* bar) { pthread_barrier_wait((pthread_barrier_t*)bar); }
}}

template <class T>
static T ld(const uint32_t* p) { T x; memcpy(&x, p, sizeof(T)); return x; }
template <class T>
static void st(uint32_t* p, const T& x) { memcpy(p, &x, sizeof(T)); }

template <class F, class Fn>
static void run_xt(Fn fn) {
  constexpr int L = xt::TeamOf<F>::LANES;
  std::vector<uint32_t> bus(2 * xt::TeamOf<F>::BUS_WORDS + sizeof(Aff<F>), 0);
  pthread_barrier_t bar;
  pthread_barrier_init(&bar, nullptr, L);
  std::vector<std::thread> th;
  for (int t = 0; t < L; t++) th.emplace_back([&, t] { xt::Team tm{t, bus.data(), 0, &bar}; fn(tm); });
  for (auto& t : th) t.join();
  pthread_barrier_destroy(&bar);
}

template <int GROUP>
static EndoSplit split_of(const uint32_t* k) {
  EndoBits b;
  endo_decompose<GROUP>(k, b);
  EndoSplit s;
  endo_split<GROUP>(b, s);
  return s;
}

// D = [2^H] p on one team (k_fold_pre), one team per part over {E^k(p), E^k(D)}, the parts brought to affine form, then
// lo + the parts on one team (k_fold4_xp<true>)
template <class F, int GROUP>
static void pre_fold(const uint32_t* p, const uint32_t* lo, const uint32_t* k, uint32_t* out) {
  constexpr int M = SplitOf<GROUP>::PARTS;
  const EndoSplit s = split_of<GROUP>(k);
  Aff<F> d;
  run_xt<F>([&](const xt::Team& tm) {
    Aff<F> r = xt::pow2_mul<F>(tm, ld<Aff<F>>(p), SplitOf<GROUP>::H);
    if (tm.t == 0) d = r;
  });
  std::vector<Aff<F>> parts(M);
  for (int part = 0; part < M; part++)
    run_xt<F>([&](const xt::Team& tm) {
      const Aff<F> src = (part & 1) ? d : ld<Aff<F>>(p);
      Jac<F> acc = xt::naf_mul_endo<F>(tm, src, M / 2, part >> 1, s.pos[part], s.neg[part], s.nbits[part],
                                       tm.bus + 2 * xt::TeamOf<F>::BUS_WORDS);
      Aff<F> pa = xt::to_affine<F>(tm, acc);
      if (tm.t == 0) parts[part] = pa;
    });
  run_xt<F>([&](const xt::Team& tm) {
    Jac<F> sum = Jac<F>::from_affine(ld<Aff<F>>(lo));
    for (int t = 0; t < M; t++) sum = xt::madd<F>(tm, sum, parts[t]);
    Aff<F> o = xt::to_affine<F>(tm, sum);
    if (tm.t == 0) st(out, o);
  });
}

extern "C" {
// out = k * p + lo (k = 8 canonical words; group 1 = G1, 2 = G2)
void hs_pre_fold(int group, const uint32_t* p, const uint32_t* lo, const uint32_t* k, uint32_t* out) {
  if (group == 1)
    pre_fold<Fq, 1>(p, lo, k, out);
  else
    pre_fold<Fq2, 2>(p, lo, k, out);
}
// the split recoding of k: out = pos[8][3] || neg[8][3] || nbits[8]
void hs_endo_split(int group, const uint32_t* k, uint32_t* out) {
  const EndoSplit s = group == 1 ? split_of<1>(k) : split_of<2>(k);
  memcpy(out, s.pos, sizeof(s.pos));
  memcpy(out + 24, s.neg, sizeof(s.neg));
  for (int t = 0; t < 8; t++) out[48 + t] = (uint32_t)s.nbits[t];
}
}
