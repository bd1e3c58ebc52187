// Shared host-side plumbing of the library: context, error reporting, launch accounting.
#pragma once
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>

#include <string>
#include <vector>

#include "../../include/ripp_b200.h"
#include "pairing.cuh"

using namespace ripp;

// ------------------------------------------------------------------------------------------------
// context / errors
// ------------------------------------------------------------------------------------------------
std::string& ripp_err_slot();

#define RIPP_SCRATCH_SLOTS 52
#define RIPP_MAX_BATCH 8
#define RIPP_MAX_CHILD 8
// per-category device-time accounting (CUDA events on the context's stream; off by default)
// RIPP_T_MSM = the bucket accumulation kernels of an MSM (the algorithmic work); its sort and its reduction / Horner tail
// are kernels of their own kind and are accounted separately
enum { RIPP_T_MILLER = 0, RIPP_T_FINAL_EXP, RIPP_T_MSM, RIPP_T_FOLD, RIPP_T_SCALE, RIPP_T_OTHER, RIPP_T_MSM_SORT, RIPP_T_MSM_REDUCE,
       RIPP_T_NCAT };
struct TimingRec {
  int cat;
  cudaEvent_t a, b;
};

struct ripp_ctx {
  int device;
  cudaStream_t stream;
  cudaStream_t own_stream;
  uint64_t launches;
  int timing;
  std::vector<TimingRec>* recs;
  // child contexts (own stream + scratch, same device) for work that may overlap on the GPU
  ripp_ctx* child[RIPP_MAX_CHILD];
  ripp_ctx* parent;
  cudaEvent_t ev;
  // scratch (grown on demand)
  void* scratch[RIPP_SCRATCH_SLOTS];
  size_t scratch_bytes[RIPP_SCRATCH_SLOTS];
  // page-locked host staging for the small per-round results (a pageable cudaMemcpyAsync goes through the driver's
  // own staging buffer and blocks the calling thread)
  uint8_t* pinned;
  // multi-GPU (comm.cu): one process per GPU, an NCCL communicator owned by the top-level context
  void* comm;  // ncclComm_t
  int rank, world;
  // set (on the parent) by a GIPA recursion once its vectors are short and the GPU mostly idle: side products that are
  // not on the critical path wait for it instead of competing with the long early rounds (gipa.cu, aggregate)
  int rounds_short;
  // work nothing waits for (the aggregation's side products): the pairing engine packs it into the fewest CTAs so that
  // the lone warps of the critical path keep sub-partitions to themselves
  int background;
  // page-locked staging grown on demand: the per-round results of the batch prover (aggregate_batch.cuh)
  uint8_t* pinned_big;
  size_t pinned_big_bytes;
};
#define RIPP_PINNED_BYTES 16384

static inline int fail(int code, const std::string& msg) {
  ripp_err_slot() = msg;
  return code;
}
#define CU(call)                                                                                         \
  do {                                                                                                   \
    cudaError_t e_ = (call);                                                                             \
    if (e_ != cudaSuccess)                                                                               \
      return fail(RIPP_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_) + " @" + __FILE__ + ":" + \
                                     std::to_string(__LINE__));                                          \
  } while (0)
#define OK(call)              \
  do {                        \
    int s_ = (call);          \
    if (s_ != RIPP_OK) return s_; \
  } while (0)
#define LAUNCHED(ctx)        \
  do {                       \
    (ctx)->launches++;       \
    CU(cudaGetLastError());  \
  } while (0)

static inline int scratch(ripp_ctx* ctx, int slot, size_t bytes, void** out) {
  if (ctx->scratch_bytes[slot] < bytes) {
    if (ctx->scratch[slot]) CU(cudaFree(ctx->scratch[slot]));
    ctx->scratch[slot] = nullptr;
    ctx->scratch_bytes[slot] = 0;
    CU(cudaMalloc(&ctx->scratch[slot], bytes));
    ctx->scratch_bytes[slot] = bytes;
  }
  *out = ctx->scratch[slot];
  return RIPP_OK;
}


static inline int pinned(ripp_ctx* ctx, uint8_t** out) {
  if (!ctx->pinned) CU(cudaHostAlloc((void**)&ctx->pinned, RIPP_PINNED_BYTES, cudaHostAllocDefault));
  *out = ctx->pinned;
  return RIPP_OK;
}

struct TimeScope {
  ripp_ctx* c;
  long idx;
  TimeScope(ripp_ctx* ctx, int cat) : c(ctx), idx(-1) {
    if (!c->timing || !c->recs) return;
    TimingRec r;
    r.cat = cat;
    if (cudaEventCreate(&r.a) != cudaSuccess || cudaEventCreate(&r.b) != cudaSuccess) return;
    cudaEventRecord(r.a, c->stream);
    c->recs->push_back(r);
    idx = (long)c->recs->size() - 1;
  }
  ~TimeScope() {
    if (idx >= 0) cudaEventRecord((*c->recs)[idx].b, c->stream);
  }
};

// cross-file internals
ripp_ctx* ripp_child(ripp_ctx* ctx, int idx);          // lazily created; NULL on failure
int ripp_fork(ripp_ctx* ctx, ripp_ctx* child);         // child's stream waits for everything queued on ctx's
int ripp_join(ripp_ctx* ctx, ripp_ctx* child);         // ctx's stream waits for everything queued on child's
int ripp_pairing_batch_l6(ripp_ctx* ctx, int nseg, const void* const* g1, const void* const* g2, size_t n, void* out,
                          bool with_final_exp);
int ripp_final_exp_l6(ripp_ctx* ctx, const void* in, uint32_t T, void* out, int nseg);
int ripp_gt_multiexp_l6(ripp_ctx* ctx, const void* in, const void* sc, size_t n, void* out, int nseg = 1);
int ripp_gt_check_l6(ripp_ctx* ctx, const void* in, size_t n, uint32_t* bad_dev, uint32_t flag, const uint32_t* owner_dev = nullptr);
// the aggregate verifier's pairing equations (verify_batch.cuh): p, q are 3 x n pairs, tgt n targets, ok n verdicts
int ripp_pairing_checks_l6(ripp_ctx* ctx, const void* p, const void* q, size_t n, void* miller, const void* tgt, uint8_t* ok);
// comm.cu: all-gather of one `bytes`-sized blob per rank on ctx's stream (recv = world * bytes, rank order); world == 1 copies
int ripp_all_gather_internal(ripp_ctx* ctx, const void* send_dev, size_t bytes, void* recv_dev);
void ripp_comm_release(ripp_ctx* ctx);
// msm.cu: the (up to four) folds of one GIPA round in ONE launch when the vectors are short enough for lane teams;
// with `pre` (written by ripp_fold_pre_internal, for vectors up to ripp_fold_pre_max_n()) over precomputed bases
int ripp_fold4_internal(ripp_ctx* ctx, const int* types, const void* const* hi, const void* const* lo, const void* const* cs, size_t n,
                        void* const* out, int* fused, const void* const* pre = nullptr);
int ripp_fold_pre_internal(ripp_ctx* ctx, const int* types, const void* const* hi, size_t n, void* const* pre);
size_t ripp_fold_pre_max_n();
// the folds of the lock-step batch prover (aggregate_batch.cuh): section s (0 G1, 1 G2, 2 Fr) has ngroups[s] groups of K
// jobs; job (g, k) folds base[s][g] + k stride[s][g] (hi at + n elements) with scalar record sc[s][g][k] (device: EndoBits
// for G1 / G2, Fr for Fr).  bpj / first_block / blocks are filled by ripp_fold_table_internal.
struct FoldTable {
  char* base[3][3];
  size_t stride[3][3];
  const void* sc[3][3];
  int ngroups[3];
  uint32_t K, n;
  uint32_t bpj[3], first_block[3], blocks[3];
};
int ripp_fold_table_internal(ripp_ctx* ctx, FoldTable t);
namespace ripp {
struct EndoBits;
}
void ripp_endo_bits(int group, const void* fr_mont_host, EndoBits* out);  // group 1 / 2: the fold recoding of a G1 / G2 scalar
int ripp_msm_batch_internal(ripp_ctx* ctx, int group, const void* bases, size_t bases_stride, const void* sc, size_t sc_stride,
                            size_t n, size_t nseg, void* out);
// nseg pairing products of n pairs each, segment s = (segs[2s], segs[2s+1]) (G1, G2 device pointers, read from device
// memory); out[s] = final_exponentiation(prod e(P_i, Q_i))
int ripp_pairing_table_l6(ripp_ctx* ctx, const void* segs_dev, size_t nseg, size_t n, void* out, int slot0);
int ripp_pairing6_init_device();  // per-device kernel attributes; called by ripp_ctx_create with the device current
// groth16.cu's kernels: fixed-base tables and prepare_inputs (setup.cu), Miller loops and checks (pairing6.cu)
size_t ripp_groth16_table_bytes();  // one input's table
int ripp_groth16_tables(ripp_ctx* ctx, const void* ic_dev, size_t m, void* tables_dev);
int ripp_groth16_inputs(ripp_ctx* ctx, const void* ic0_dev, const void* tables_dev, size_t m, const void* x_dev, size_t n,
                        void* out_dev);
int ripp_groth16_pairings_l6(ripp_ctx* ctx, const void* a, const void* b, const void* p, const void* c, const void* neg_gamma,
                             const void* neg_delta, const void* ab, size_t n, void* miller, const uint8_t* pre, uint8_t* out);
// the segment checks of the random-linear-combination entry points: ok[t] = 1 / 0 for segment t < nseg of s proofs
int ripp_groth16_rlc_pairings_l6(ripp_ctx* ctx, const void* ra, const void* b, const void* ps, const void* cs, const void* neg_gamma,
                                 const void* neg_delta, const void* ab, size_t n, size_t s, size_t nseg, uint8_t* ok);
// deserialize.cu: one H2D copy of n proof records (plus `extra` bytes of the caller's behind them), A, B, C decoded on
// three streams; statuses S[0, n) A, [n, 2n) B, [2n, 3n) C
struct DecodedProofs {
  void *a, *b, *c, *extra;
  uint8_t* status;
};
int ripp_decode_proofs(ripp_ctx* ctx, const uint8_t* proofs_host, size_t n, int compressed, size_t extra, DecodedProofs* out);
