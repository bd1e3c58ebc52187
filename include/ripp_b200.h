/* ripp_b200 -- C ABI of the B200-native backend for RIPP's inner-pairing-product hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b): a thin Rust crate implements the reference's
 * traits by calling these entry points (binding sketch in INTEGRATION.md).  Each function cites
 * the reference interface it replaces (paths relative to the arkworks-rs/ripp checkout).
 * There is no CPU fallback: every compute entry point launches CUDA kernels or fails.
 *
 * Data layout (all little-endian, packed, no padding):
 *   Fr   : 8  x u32  Montgomery form, R = 2^256   (== ark-ff Fp256 limbs, [u64; 4])
 *   Fq   : 12 x u32  Montgomery form, R = 2^384   (== ark-ff Fp384 limbs, [u64; 6])
 *   Fq2  : c0, c1
 *   G1 affine   : x, y            (96 B)   identity = all-zero bytes
 *   G2 affine   : x, y over Fq2   (192 B)  identity = all-zero bytes
 *   G1 Jacobian : X, Y, Z         (144 B)  == ark-ec short_weierstrass::Projective; identity Z = 0
 *   G2 Jacobian : X, Y, Z         (288 B)
 *   GT   : Fq12 = c0.c0, c0.c1, c0.c2, c1.c0, c1.c1, c1.c2 (each Fq2) (576 B) == ark PairingOutput.0
 *
 * Status: 0 = ok; negative = ripp_status.  ripp_last_error_string() describes the last failure
 * on the calling thread.  Entry points taking `_dev` pointers expect device memory of the
 * context's GPU and are asynchronous on the context's stream unless they return host data.
 */
#ifndef RIPP_B200_H
#define RIPP_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum ripp_status {
  RIPP_OK = 0,
  RIPP_ERR_LEN_MISMATCH = -1, /* InnerProductError::MessageLengthInvalid, inner_products/src/lib.rs:18-38 */
  RIPP_ERR_NOT_POW2 = -2,     /* gipa.rs:116-122,140-146 */
  RIPP_ERR_CUDA = -3,
  RIPP_ERR_ARG = -4,
  RIPP_ERR_INNER_PRODUCT = -5, /* InnerProductArgumentError::InnerProductInvalid, ip_proofs/src/lib.rs:22-25 */
  RIPP_ERR_NO_DEVICE = -6,
  RIPP_ERR_NCCL = -7          /* NCCL could not be loaded, or a collective failed */
} ripp_status;

typedef struct ripp_ctx ripp_ctx;

/* ---- context ---------------------------------------------------------------------------- */
/* One context per GPU / per process rank.  `device` is the CUDA ordinal. */
int ripp_ctx_create(int device, ripp_ctx** out);
void ripp_ctx_destroy(ripp_ctx* ctx);
const char* ripp_last_error_string(void);
/* Blocks until all work queued on the context's stream has finished. */
int ripp_ctx_sync(ripp_ctx* ctx);
/* cudaStream_t of the context (as void*), for callers that time with CUDA events. */
void* ripp_ctx_stream(ripp_ctx* ctx);
/* Run on a caller-owned stream instead (e.g. torch's current stream, so that NCCL collectives and
 * CUDA-event timing issued by the host framework are ordered with this library's kernels). */
int ripp_ctx_set_stream(ripp_ctx* ctx, void* cuda_stream);
/* Number of kernels launched by this context so far (bench.py's gpu_launches). */
uint64_t ripp_ctx_launch_count(ripp_ctx* ctx);

/* Per-category device-time accounting with CUDA events on the context's stream (off by default).
 * Categories: 0 Miller loops (+ Fq12 product tree), 1 final exponentiations, 2 MSM bucket accumulation, 3 folds,
 * 4 element-wise scalar muls, 5 other, 6 MSM digit recoding / sort, 7 MSM bucket reduction + window sums + Horner tail.
 * ripp_ctx_timing synchronises, returns the sums since the last call (arrays of 8) and resets them. */
int ripp_ctx_set_timing(ripp_ctx* ctx, int on);
int ripp_ctx_timing(ripp_ctx* ctx, double* ms_by_cat, uint64_t* count_by_cat);

/* ---- device memory (residency; SURVEY.md §8b "residency") -------------------------------- */
int ripp_dev_alloc(ripp_ctx* ctx, size_t bytes, void** dev_out);
int ripp_dev_free(ripp_ctx* ctx, void* dev);
int ripp_dev_upload(ripp_ctx* ctx, void* dev_dst, const void* host_src, size_t bytes);
int ripp_dev_download(ripp_ctx* ctx, void* host_dst, const void* dev_src, size_t bytes);

/* ---- L1: inner products (inner_products/src/lib.rs) --------------------------------------- */
/* PairingInnerProduct::inner_product (lib.rs:56-74) == cfg_multi_pairing (lib.rs:77-116):
 * out = prod_i e(left[i], right[i]).  Host pointers, Jacobian inputs exactly as arkworks holds
 * them; normalisation (lib.rs:80-81) happens on the GPU.  n_left != n_right -> LEN_MISMATCH. */
int ripp_pairing_ip(ripp_ctx* ctx, const void* g1_jac, size_t n_left, const void* g2_jac, size_t n_right,
                    void* gt_out);
/* Same product over packed affine host inputs (sipp/src/lib.rs:221-224 product_of_pairings). */
int ripp_pairing_ip_affine(ripp_ctx* ctx, const void* g1_aff, size_t n_left, const void* g2_aff, size_t n_right,
                           void* gt_out);
/* Device-resident variant: affine device vectors, result written to device memory (576 B). */
int ripp_pairing_ip_dev(ripp_ctx* ctx, const void* g1_aff_dev, const void* g2_aff_dev, size_t n, void* gt_out_dev);
/* Several equal-length products in ONE launch (the six commitments of a GIPA round, gipa.rs:220-231):
 * g1_aff_dev / g2_aff_dev are HOST arrays of nseg (<= 8) device pointers; out gets nseg GT values. */
int ripp_pairing_ip_batch_dev(ripp_ctx* ctx, int nseg, const void* const* g1_aff_dev, const void* const* g2_aff_dev,
                              size_t n, void* gt_out_dev);
/* Sharded variant for multi-GPU (SURVEY.md §8e): product of Miller-loop values of this rank's
 * slice WITHOUT the final exponentiation (one Fq12 partial, device memory) ... */
int ripp_miller_partial_dev(ripp_ctx* ctx, const void* g1_aff_dev, const void* g2_aff_dev, size_t n,
                            void* fq12_out_dev);
/* ... and the combine: multiply `count` partials (gathered from all ranks, device memory) and
 * apply the single shared final exponentiation (lib.rs:115). */
int ripp_gt_combine_dev(ripp_ctx* ctx, const void* fq12_partials_dev, size_t count, void* gt_out_dev);

/* Batch forms for the sharded provers (DESIGN.md §5; SURVEY.md §8e "GIPA rounds"): the six products of a GIPA
 * round (gipa.rs:220-231) over this rank's share in ONE Miller launch, no final exponentiation ... */
int ripp_miller_partial_batch_dev(ripp_ctx* ctx, int nseg, const void* const* g1_aff_dev, const void* const* g2_aff_dev,
                                  size_t n, void* fq12_out_dev);
/* ... and out[s] = final_exponentiation(prod_r partials[s * count + r]) for the gathered per-rank partials. */
int ripp_gt_combine_batch_dev(ripp_ctx* ctx, const void* fq12_partials_dev, size_t count, int nseg, void* gt_out_dev);
/* out[s] = sum_r in[s * count + r]: per-rank MSM / scalar partials added in rank order.
 * type: 1 = G1 affine, 2 = G2 affine, 3 = Fr. */
int ripp_seg_sum_dev(ripp_ctx* ctx, int type, const void* in_dev, size_t count, int nseg, void* out_dev);

/* MultiexponentiationInnerProduct::inner_product (lib.rs:123-142) == G::msm(normalize_batch(left), right),
 * also PedersenCommitment::commit (dh_commitments/src/pedersen/mod.rs:24-26).  Host pointers:
 * bases Jacobian, scalars Fr (Montgomery), result Jacobian (Z = 1, or Z = 0 for the identity). */
int ripp_msm_g1(ripp_ctx* ctx, const void* g1_jac, size_t n_left, const void* fr, size_t n_right, void* g1_jac_out);
int ripp_msm_g2(ripp_ctx* ctx, const void* g2_jac, size_t n_left, const void* fr, size_t n_right, void* g2_jac_out);
/* Device-resident variants: affine bases, result one affine point in device memory.  Also the
 * KZG opening MSM of tipa/mod.rs:333-334. */
int ripp_msm_g1_dev(ripp_ctx* ctx, const void* g1_aff_dev, const void* fr_dev, size_t n, void* g1_aff_out_dev);
int ripp_msm_g2_dev(ripp_ctx* ctx, const void* g2_aff_dev, const void* fr_dev, size_t n, void* g2_aff_out_dev);
/* nseg MSMs of n terms in one segmented pass: out[s] = sum_i fr[s*n + i] * bases[s*bases_stride + i], s < nseg (device
 * memory, affine bases, Montgomery scalars, nseg affine results).  bases_stride = 0: one base vector shared by all
 * segments (KZG openings over one SRS).  nseg at most 2^16 and nseg * n at most 2^24 (RIPP_ERR_ARG): a short segment
 * needs ~65 KB of workspace (G2), a long one about what one MSM over all nseg * n points needs. */
int ripp_msm_g1_batch_dev(ripp_ctx* ctx, const void* g1_aff_dev, size_t bases_stride, const void* fr_dev, size_t n, size_t nseg,
                          void* g1_aff_out_dev);
int ripp_msm_g2_batch_dev(ripp_ctx* ctx, const void* g2_aff_dev, size_t bases_stride, const void* fr_dev, size_t n, size_t nseg,
                          void* g2_aff_out_dev);
/* ScalarInnerProduct::inner_product (lib.rs:149-166): sum_i a[i] * b[i] in Fr. */
int ripp_scalar_ip(ripp_ctx* ctx, const void* fr_a, size_t n_left, const void* fr_b, size_t n_right, void* fr_out);
int ripp_scalar_ip_dev(ripp_ctx* ctx, const void* fr_a_dev, const void* fr_b_dev, size_t n, void* fr_out_dev);

/* ---- folds with one shared scalar (kernel K7) ------------------------------------------------ */
/* out[i] = hi[i] * c + lo[i]: the four "rescale" maps of a GIPA round (gipa.rs:261-291, scalar-mul
 * primitive mul_helper, ip_proofs/src/lib.rs:15-19) and of SIPP (sipp/src/lib.rs:87-100).
 * c is ONE Fr in Montgomery form in HOST memory (32 B); vectors are device-resident (affine points
 * or Fr); out may alias lo.  Only the significant bits of c are walked, so the 128-bit challenges
 * cost half of a full-width scalar. */
int ripp_g1_fold_dev(ripp_ctx* ctx, const void* hi_dev, const void* lo_dev, const void* c_host, size_t n, void* out_dev);
int ripp_g2_fold_dev(ripp_ctx* ctx, const void* hi_dev, const void* lo_dev, const void* c_host, size_t n, void* out_dev);
int ripp_fr_fold_dev(ripp_ctx* ctx, const void* hi_dev, const void* lo_dev, const void* c_host, size_t n, void* out_dev);

/* ---- element-wise scalar multiplication (kernel K8) ------------------------------------------ */
/* out[i] = scalars[i] * points[i] with distinct scalars: the `a[i] * r^i` / `ck[i] * r^-i` maps of
 * groth16_aggregation.rs:118-131 and `a[i] * r[i]` of sipp/src/lib.rs:61-65,189-193.
 * points == NULL means the standard generator for every i (tipa/mod.rs:153-160 SRS powers and the
 * synthetic inputs of SURVEY.md §8d).  Scalars are Fr in Montgomery form; inputs/outputs affine,
 * device memory. */
int ripp_g1_scale_dev(ripp_ctx* ctx, const void* g1_aff_dev, const void* fr_dev, size_t n, void* g1_aff_out_dev);
int ripp_g2_scale_dev(ripp_ctx* ctx, const void* g2_aff_dev, const void* fr_dev, size_t n, void* g2_aff_out_dev);

/* ---- setup (SURVEY.md §8 rows a9, a14) ----------------------------------------------------------- */
/* The random draws of the reference's setups (Fr::rand / G::rand on the caller's Rng) stay with the caller; these
 * entry points take the exponents, so the Rust shim keeps arkworks' own random stream (INTEGRATION.md "setup").
 *
 * ark-ec FixedBase::msm over ONE base as structured_generators_scalar_power uses it (tipa/mod.rs:384-389):
 * out[i] = s[i] * base.  base: one affine point (host, Montgomery) or NULL for the standard generator; s: n Fr
 * (device, Montgomery); out: n affine points (device).  With s[i] drawn by the caller this is also the key vector
 * of random_generators (dh_commitments/src/lib.rs:59-61) for the synthetic keys of SURVEY.md §8d. */
int ripp_fixed_base_msm_g1_dev(ripp_ctx* ctx, const void* base_g1_aff, const void* fr_dev, size_t n, void* g1_aff_out_dev);
int ripp_fixed_base_msm_g2_dev(ripp_ctx* ctx, const void* base_g2_aff, const void* fr_dev, size_t n, void* g2_aff_out_dev);
/* structured_generators_scalar_power (tipa/mod.rs:372-391): out[i] = s^i * base, i < num (num > 0 as :377 asserts).
 * s: one Fr (host, Montgomery). */
int ripp_structured_generators_g1_dev(ripp_ctx* ctx, const void* base_g1_aff, const void* s, size_t num, void* g1_aff_out_dev);
int ripp_structured_generators_g2_dev(ripp_ctx* ctx, const void* base_g2_aff, const void* s, size_t num, void* g2_aff_out_dev);
/* TIPA::setup (tipa/mod.rs:150-164) for given trapdoors alpha, beta (host Fr, Montgomery): the 2 size - 1 powers
 * g^(alpha^i) and h^(beta^i) stay on the device (they are the long-lived SRS of the provers above), g^beta and
 * h^alpha (the rest of VerifierSRS, tipa/mod.rs:120-127) come back to the host as affine points. */
int ripp_tipa_setup_dev(ripp_ctx* ctx, const void* alpha, const void* beta, size_t size, void* srs_g1_out_dev,
                        void* srs_g2_out_dev, void* g_beta_out, void* h_alpha_out);

/* ---- L3: device-resident provers ------------------------------------------------------------ */
/* Instantiations of GIPA<IP, LMC, RMC, IPC, Blake2b> (ip_proofs/src/gipa.rs:16-22); element types of
 * (left message A, right message B, left key v, right key w): */
typedef enum ripp_gipa_kind {
  RIPP_GIPA_PAIRING = 0,               /* Pairing, AFGHO-G1, AFGHO-G2, Identity<GT>: (G1, G2, G2, G1)   gipa.rs:472-475 */
  RIPP_GIPA_MULTIEXP_PEDERSEN = 1,     /* Multiexp<G1>, AFGHO-G1, Pedersen<G1>, Identity<G1>: (G1, Fr, G2, G1)  gipa.rs:500-503 */
  RIPP_GIPA_MULTIEXP_SSM = 2,          /* Multiexp<G1>, AFGHO-G1, SSMPlaceholder, Identity<G1>: (G1, Fr, G2, -)
                                          structured_scalar_message.rs:130-136, groth16_aggregation.rs:42-48 */
  RIPP_GIPA_SCALAR_PEDERSEN_G2_G2 = 3, /* Scalar, Pedersen<G2>, Pedersen<G2>, Identity<Fr>: (Fr, Fr, G2, G2)  gipa.rs:531-536 */
  RIPP_GIPA_SCALAR_PEDERSEN_G2_G1 = 4, /* Scalar, Pedersen<G2>, Pedersen<G1>, Identity<Fr>: (Fr, Fr, G2, G1)  tipa/mod.rs:501-506 */
  RIPP_GIPA_SCALAR_SSM = 5,            /* Scalar, Pedersen<G2>, SSMPlaceholder, Identity<Fr>: (Fr, Fr, G2, -)
                                          structured_scalar_message.rs:392-423 */
  RIPP_GIPA_SCALAR_SSM_G1 = 6          /* Scalar, Pedersen<G1>, SSMPlaceholder, Identity<Fr>: (Fr, Fr, G1, -)
                                          the first-tier argument of applications/poly_commit/transparent.rs:44-49 */
} ripp_gipa_kind;

/* GIPA::prove_with_aux (gipa.rs:162-178 -> _prove :181-312).  Vectors are device resident (affine
 * points / Fr), n a power of two; they are not modified.  Runs all log2(n) rounds on the device.
 *   proof_out      GIPAProof in arkworks serialize_uncompressed bytes (steps reversed as gipa.rs:298-299,
 *                  then r_base); *proof_len receives the length (also when proof_cap is too small)
 *   transcript_out log2(n) Fr (Montgomery): GIPAAux::r_transcript, may be NULL
 *   ck_base_out    GIPAAux::ck_base = (v0, w0) serialised */
int ripp_gipa_prove_dev(ripp_ctx* ctx, int kind, const void* a_dev, const void* b_dev, const void* v_dev,
                        const void* w_dev, size_t n, uint8_t* proof_out, size_t proof_cap, size_t* proof_len,
                        void* transcript_out, uint8_t* ck_base_out, size_t ck_cap, size_t* ck_len);

/* GIPA::prove (gipa.rs:108-133), the CHECKED entry: recomputes IP(l, r), LMC::commit(ck_a, l) and RMC::commit(ck_b, r)
 * on the device and compares them with the caller's statement before proving.  `com` is the statement in the
 * verifier's layout (see ripp_gipa_verify_dev): com_a || com_b || com_t, no com_b for the *_SSM kinds.
 * RIPP_ERR_INNER_PRODUCT = InnerProductArgumentError::InnerProductInvalid (wrong inner product, or a commitment
 * that does not open to the message); RIPP_ERR_NOT_POW2 = MessageLengthInvalid -- checked in the reference's order. */
int ripp_gipa_prove_checked_dev(ripp_ctx* ctx, int kind, const void* a_dev, const void* b_dev, const void* v_dev,
                                const void* w_dev, size_t n, const uint8_t* com, size_t com_len, uint8_t* proof_out,
                                size_t proof_cap, size_t* proof_len);

/* The same prover continuing a transcript: prev_challenge (one Fr, host, Montgomery) is the challenge of the round
 * before the first one proved here (NULL = fresh transcript, i.e. ripp_gipa_prove_dev).  A sharded prover
 * (ripp_b200/parallel.py) runs its long rounds partitioned over the GPUs, all-gathers the short remaining vectors
 * and hands this tail -- latency-bound, replicated on every rank -- to the resident single-GPU prover.  The proof
 * bytes cover the rounds proved here: u64 count, their steps (last round first), then r_base. */
int ripp_gipa_prove_resume_dev(ripp_ctx* ctx, int kind, const void* a_dev, const void* b_dev, const void* v_dev,
                               const void* w_dev, size_t n, const void* prev_challenge, uint8_t* proof_out,
                               size_t proof_cap, size_t* proof_len, void* transcript_out, uint8_t* ck_base_out,
                               size_t ck_cap, size_t* ck_len);

/* prove_commitment_key_kzg_opening (tipa/mod.rs:304-337): opening of the product-form polynomial
 * f(X) = prod_j (1 + x_j r^(2^j) X^(2^(j+1))) at z over n_srs = 2*2^k - 1 SRS powers (device).
 * transcript (k Fr), r_shift, z: host, Montgomery.  Result: one affine point (host). */
int ripp_kzg_open_g1_dev(ripp_ctx* ctx, const void* srs_g1_dev, size_t n_srs, const void* transcript, size_t k,
                         const void* r_shift, const void* z, void* g1_aff_out);
int ripp_kzg_open_g2_dev(ripp_ctx* ctx, const void* srs_g2_dev, size_t n_srs, const void* transcript, size_t k,
                         const void* r_shift, const void* z, void* g2_aff_out);

/* The quotient coefficients q = (f - f(z)) / (X - z) of the opening above (tipa/mod.rs:313-332), host in / host
 * out (n_srs Fr, Montgomery, zero padded): with them every rank of a sharded prover runs the opening MSM over its
 * own slice of the SRS powers and the partial points are summed (SURVEY.md §8e "KZG openings"). */
int ripp_kzg_quotient(const void* transcript, size_t k, const void* r_shift, const void* z, size_t n_srs, void* fr_out);

/* TIPA::prove_with_srs_shift (tipa/mod.rs:176-231) for kinds with a G1 right key, and
 * TIPAWithSSM::prove_with_structured_scalar_message (structured_scalar_message.rs:211-268) for the
 * *_SSM kinds (w_dev NULL, r_shift ignored).  srs_g1 = g^(alpha^i), srs_g2 = h^(beta^i), i < 2n-1.
 * r_shift: one Fr (host, Montgomery) or NULL for 1.  Output: TIPAProof / TIPAWithSSMProof bytes. */
int ripp_tipa_prove_dev(ripp_ctx* ctx, int kind, const void* srs_g1_dev, const void* srs_g2_dev, const void* a_dev,
                        const void* b_dev, const void* v_dev, const void* w_dev, size_t n, const void* r_shift,
                        uint8_t* proof_out, size_t proof_cap, size_t* proof_len);

/* ---- L4: aggregate_proofs (applications/groth16_aggregation.rs:77-160) ------------------------ */
/* a, c: n G1 affine; b: n G2 affine (the Groth16 proofs' A, B, C); SRS as above.  Output bytes:
 * com_a, com_b, com_c, ip_ab (GT), agg_c (G1), TIPAProof(ab), TIPAWithSSMProof(c) -- the field order
 * of AggregateProof (:58-66).  Fails with RIPP_ERR_INNER_PRODUCT if the :133-136 assertion fails. */
int ripp_tipp_aggregate_dev(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, const void* a_dev,
                            const void* b_dev, const void* c_dev, size_t n, uint8_t* proof_out, size_t proof_cap,
                            size_t* proof_len);

/* aggregate_proofs with the Groth16 proofs in HOST memory, exactly as arkworks holds
 * `Proof { a: G1Affine, b: G2Affine, c: G1Affine }` split into three packed arrays (n x 96 B, n x 192 B,
 * n x 96 B); the SRS is long-lived and stays device resident.  This is the end-to-end entry point
 * bench.py times (H2D of the proofs + all kernels + D2H of the proof bytes). */
int ripp_tipp_aggregate(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, const void* a_host,
                        const void* b_host, const void* c_host, size_t n, uint8_t* proof_out, size_t proof_cap,
                        size_t* proof_len);

/* aggregate_proofs for `count` independent batches of n proofs each, under one SRS (at least 2n - 1 powers, as
 * ripp_tipp_aggregate_dev).  a, c: count x n G1 affine, b: count x n G2 affine, batch k at element k * n.  proofs_out
 * receives count AggregateProofs back to back, each *proof_len bytes (the length depends on n only), and proof k is
 * byte for byte what ripp_tipp_aggregate_dev returns for batch k alone.  The GIPA rounds of all batches run in lock
 * step: the number of launches and host synchronisations does not grow with count.
 * n: a power of two (RIPP_ERR_NOT_POW2), at least 2 (RIPP_ERR_ARG); count == 0: RIPP_OK with *proof_len = 0;
 * count * n at most 2^20 and count at most 2^16 (RIPP_ERR_ARG; the device workspace then stays below ~41 GB, kept on
 * the context for the next call); proofs_cap < count * *proof_len: RIPP_ERR_ARG with *proof_len set.
 * RIPP_ERR_INNER_PRODUCT names the batch whose :133-136 self-check failed. */
int ripp_tipp_aggregate_batch_dev(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, size_t count, size_t n,
                                  const void* a_dev, const void* b_dev, const void* c_dev, uint8_t* proofs_out,
                                  size_t proofs_cap, size_t* proof_len);
/* Same with the proofs in host memory (three packed arrays, one H2D copy each), as ripp_tipp_aggregate. */
int ripp_tipp_aggregate_batch(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, size_t count, size_t n,
                              const void* a_host, const void* b_host, const void* c_host, uint8_t* proofs_out,
                              size_t proofs_cap, size_t* proof_len);

/* ---- deserialisation: validated decoding of untrusted ark-serialize bytes ------------------------------------ */
/* Points as ark-serialize 0.4 / ark-bls12-381 0.4 write them (big-endian coordinates, flags in the top three bits
 * of byte 0: 0x80 compressed, 0x40 infinity, 0x20 lexicographically largest y).  G1: x (48 B) or x || y (96 B);
 * G2: x.c1 || x.c0 (96 B) or x.c1 || x.c0 || y.c1 || y.c0 (192 B).  Decoding validates what deserialize_* with
 * Validate::Yes validates -- flags, canonical field encoding, curve membership (a square root for compressed points,
 * the root picked by the sort flag), membership of the prime-order subgroup -- on the GPU, one thread per element.
 * Each element gets one status byte: the first check it fails, in the order of ripp_decode_status. */
typedef enum ripp_decode_status {
  RIPP_DECODE_OK = 0,
  RIPP_DECODE_FLAGS = 1,           /* compression bit != mode; sort bit without compression or with infinity;
                                      infinity with any other bit set */
  RIPP_DECODE_NONCANONICAL = 2,    /* a coordinate >= p */
  RIPP_DECODE_NOT_ON_CURVE = 3,    /* y^2 != x^3 + b, or (compressed) x^3 + b is not a square */
  RIPP_DECODE_NOT_IN_SUBGROUP = 4  /* on the curve, outside the prime-order subgroup */
} ripp_decode_status;

/* n elements, element i at bytes_dev + i * stride (stride >= the element's size, so the A, B, C of packed proof
 * records decode in place); compressed = 1 / 0 selects the mode.  Writes n affine points (Montgomery; all zero for
 * the identity and for every rejected element) and n status bytes.  Device memory, asynchronous on the context's
 * stream: a sharded caller decodes its own share on every rank and hands it to ripp_tipp_aggregate_sharded_dev. */
int ripp_g1_deserialize_dev(ripp_ctx* ctx, const void* bytes_dev, size_t n, size_t stride, int compressed,
                            void* g1_aff_out_dev, uint8_t* status_dev);
int ripp_g2_deserialize_dev(ripp_ctx* ctx, const void* bytes_dev, size_t n, size_t stride, int compressed,
                            void* g2_aff_out_dev, uint8_t* status_dev);

/* aggregate_proofs from the proofs' bytes: proofs_host holds n ark-groth16 `Proof { a, b, c }` records back to back,
 * each written with serialize_compressed (192 B) or serialize_uncompressed (384 B), no Vec length prefix.  One H2D
 * copy, A, B and C decoded and validated on the GPU, then ripp_tipp_aggregate_dev on the decoded vectors (same bytes
 * out).  proofs_len != n x record size, n < 2 and any invalid element fail with RIPP_ERR_ARG, a length that is not a
 * power of two with RIPP_ERR_NOT_POW2 -- all before any proving kernel is queued; the message of an invalid element
 * names the first bad proof, its component and the status, e.g. "proof 17: B not in the prime-order subgroup". */
int ripp_tipp_aggregate_serialized(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, const uint8_t* proofs_host,
                                   size_t proofs_len, size_t n, int compressed, uint8_t* proof_out, size_t proof_cap,
                                   size_t* proof_len);

/* ---- Groth16 verification: one verdict per proof ---------------------------------------------------------------- */
/* ark-groth16 0.4 prepare_verifying_key / prepare_inputs / verify_proof for batches: proof i is accepted iff
 *   final_exp(multi_miller_loop([A_i, P_i, C_i], [B_i, -gamma, -delta])) == e(alpha, beta),
 *   P_i = IC_0 + sum_j x_ij IC_j  (IC = gamma_abc_g1).
 * Each proof costs three Miller loops sharing one accumulator and one final exponentiation on a six-lane group;
 * P_i comes from fixed-base tables (8-bit windows) of IC_1..IC_m kept in the prepared key. */
typedef enum ripp_groth16_status {
  RIPP_GROTH16_OK = 0,               /* 0..4 are the ripp_decode_status of the first bad point, in the order A, B, C */
  RIPP_GROTH16_FLAGS = 1,
  RIPP_GROTH16_NONCANONICAL = 2,
  RIPP_GROTH16_NOT_ON_CURVE = 3,
  RIPP_GROTH16_NOT_IN_SUBGROUP = 4,
  RIPP_GROTH16_INPUT_NONCANONICAL = 5, /* a public input >= r */
  RIPP_GROTH16_REJECTED = 6            /* everything decodes, the pairing equation fails */
} ripp_groth16_status;

/* Bytes of device memory a prepared key with m public inputs needs. */
size_t ripp_groth16_pvk_bytes(size_t m);
/* vk: the packed host layout of ripp_tipp_verify_aggregate (alpha_g1 | beta_g2 | gamma_g2 | delta_g2 |
 * gamma_abc_g1[m + 1]; Montgomery, trusted).  Writes e(alpha, beta), -gamma, -delta, IC_0 and the fixed-base tables of
 * IC_1..IC_m into pvk_dev (ripp_groth16_pvk_bytes(m) bytes the caller allocated, e.g. with ripp_dev_alloc); returns
 * when the key is ready.  One key serves any number of verification calls on contexts of the same GPU. */
int ripp_groth16_prepare_vk_dev(ripp_ctx* ctx, const void* vk, size_t m, void* pvk_dev);
/* n proofs, device resident and trusted (affine Montgomery, as every other _dev entry); inputs_dev: n x m Fr
 * (Montgomery, row = one proof; NULL when m = 0).  verdict_dev[i] = 1 accept / 0 reject.  Asynchronous on the
 * context's stream. */
int ripp_groth16_verify_batch_dev(ripp_ctx* ctx, const void* pvk_dev, size_t m, const void* inputs_dev, const void* a_dev,
                                  const void* b_dev, const void* c_dev, size_t n, uint8_t* verdict_dev);
/* Untrusted bytes: proofs_host as for ripp_tipp_aggregate_serialized (n records; any n); inputs_host: n x m canonical
 * little-endian Fr (32 B each, ark-serialize, no length prefix).  status_host[i] is a ripp_groth16_status: the first
 * failure of proof i in the order A, B, C, inputs, equation.  *n_valid counts the zeros.  A false or malformed proof is
 * data, not an error: RIPP_ERR_ARG only for lengths that do not match n and m, null pointers and n > 2^32 - 1. */
int ripp_groth16_verify_serialized(ripp_ctx* ctx, const void* pvk_dev, size_t m, const uint8_t* inputs_host, size_t inputs_len,
                                   const uint8_t* proofs_host, size_t proofs_len, size_t n, int compressed,
                                   uint8_t* status_host, size_t* n_valid);
/* Random-linear-combination verification: verdicts as ripp_groth16_verify_batch_dev, except with probability
 * <= 2^-128 per segment; seed32: 32 caller-drawn bytes, fresh per call.  Synchronous (one host decision: which
 * segments to re-check).  *n_rechecked = proofs that went through the per-proof fallback.
 * Segments of s consecutive proofs (RIPP_B200_G16_RLC_SEG, default 58) are each checked as one proof whose scalars
 * r_i (ChaCha20 keystream of the seed, 128 bits, normalised to sum to one) combine the proofs' equations; the proofs
 * of a failing segment are then verified one by one (DESIGN.md §4 "Groth16 verification by random linear
 * combination"). */
int ripp_groth16_verify_rlc_dev(ripp_ctx* ctx, const void* pvk_dev, size_t m, const void* inputs_dev, const void* a_dev,
                                const void* b_dev, const void* c_dev, size_t n, const uint8_t* seed32,
                                uint8_t* verdict_dev, size_t* n_rechecked);
/* Untrusted bytes as ripp_groth16_verify_serialized, same statuses; proofs with a decode or input status are left out
 * of their segment's combination (r_i = 0, not a member) and keep that status. */
int ripp_groth16_verify_rlc_serialized(ripp_ctx* ctx, const void* pvk_dev, size_t m, const uint8_t* inputs_host,
                                       size_t inputs_len, const uint8_t* proofs_host, size_t proofs_len, size_t n,
                                       int compressed, const uint8_t* seed32, uint8_t* status_host, size_t* n_valid,
                                       size_t* n_rechecked);

/* ---- SIPP (sipp/src/lib.rs; E = BLS12-381, D = Blake2s) ---------------------------------------- */
/* product_of_pairings_with_coeffs (lib.rs:184-217): prod_i e(r_i a_i, b_i).  Affine host inputs
 * exactly as the reference takes them (&[G1Affine], &[G2Affine], &[Fr]). */
int ripp_sipp_product_with_coeffs(ripp_ctx* ctx, const void* a_aff, const void* b_aff, const void* r, size_t n,
                                  void* gt_out);
/* SIPP::prove (lib.rs:42-106).  value = the claimed product (GT, host).  proof_out receives
 * log2(n) pairs (z_l, z_r) in serialize_uncompressed form (Proof::gt_elems, lib.rs:32-34). */
int ripp_sipp_prove(ripp_ctx* ctx, const void* a_aff, const void* b_aff, const void* r, size_t n,
                    const void* value_gt, uint8_t* proof_out, size_t proof_cap, size_t* proof_len);

/* ---- multi-GPU: one process per GPU, NCCL over NVLink inside the library (SURVEY.md §8e) ------------------- */
/* The reference is single-host rayon; this is what a host behind its traits calls to span the GPUs of one box.
 * Bootstrap as NCCL itself: rank 0 calls ripp_comm_unique_id and hands the 128 bytes to every rank through whatever
 * channel the host has (MPI, a torch.distributed store, a file); every rank then calls ripp_comm_init on its
 * top-level context.  world must be a power of two.  NCCL is loaded at run time (libnccl.so.2; RIPP_B200_NCCL_LIB
 * overrides), so single-GPU users never need it.  All collectives run on the context's stream. */
int ripp_comm_unique_id(uint8_t* id128_out);
int ripp_comm_init(ripp_ctx* ctx, const uint8_t* id128, int rank, int world);
int ripp_comm_info(ripp_ctx* ctx, int* rank, int* world);
int ripp_comm_destroy(ripp_ctx* ctx);
/* all-gather of one `bytes`-sized device blob per rank (recv_dev: world * bytes, rank order) */
int ripp_all_gather_dev(ripp_ctx* ctx, const void* send_dev, size_t bytes, void* recv_dev);

/* Leaf inner products of ONE instance whose inputs are sharded by CONTIGUOUS slices (cfg_multi_pairing's chunks,
 * inner_products/src/lib.rs:91-113, spread over GPUs instead of threads): every rank computes the partial of its
 * slice (Miller value before the final exponentiation / one point), ONE all-gather of 576 / 96 / 192 bytes per
 * rank, combination in rank order and (pairing) one final exponentiation on every rank.  Same result on all ranks,
 * bit-identical to the single-GPU entry points. */
int ripp_pairing_ip_sharded_dev(ripp_ctx* ctx, const void* g1_slice_dev, const void* g2_slice_dev, size_t n_local,
                                void* gt_out_dev);
int ripp_msm_g1_sharded_dev(ripp_ctx* ctx, const void* g1_slice_dev, const void* fr_slice_dev, size_t n_local,
                            void* g1_aff_out_dev);
int ripp_msm_g2_sharded_dev(ripp_ctx* ctx, const void* g2_slice_dev, const void* fr_slice_dev, size_t n_local,
                            void* g2_aff_out_dev);

/* GIPA::prove_with_aux (gipa.rs:162-312) for ONE instance whose four vectors are partitioned CYCLICALLY: rank k holds
 * global indices j * world + k at local index j (n_local = n / world elements, a power of two).  Rounds run
 * partitioned -- local products and folds, one all-gather of six partials per round -- while the global length exceeds
 * tail_len (0 = default 2^12); the rest is gathered once and finished by the resident prover on every rank.  Outputs as
 * ripp_gipa_prove_dev, identical on all ranks and to one GPU. */
int ripp_gipa_prove_sharded_dev(ripp_ctx* ctx, int kind, const void* a_dev, const void* b_dev, const void* v_dev,
                                const void* w_dev, size_t n_local, size_t tail_len, uint8_t* proof_out, size_t proof_cap,
                                size_t* proof_len, void* transcript_out, uint8_t* ck_base_out, size_t ck_cap, size_t* ck_len);

/* aggregate_proofs (groth16_aggregation.rs:77-160) for ONE batch of n_total proofs partitioned cyclically over the
 * ranks: a, b, c are this rank's shares (n_total / world elements); the SRS (2 n_total - 1 powers each) is resident
 * in full on every rank.  The two TIPA recursions advance in lock step (one all-gather of twelve partials per
 * round), their latency-bound tails finish concurrently, the KZG opening MSMs are sharded by contiguous slices of the
 * SRS powers.  Output: the AggregateProof bytes ripp_tipp_aggregate_dev emits, on every rank. */
int ripp_tipp_aggregate_sharded_dev(ripp_ctx* ctx, const void* srs_g1_dev, const void* srs_g2_dev, const void* a_dev,
                                    const void* b_dev, const void* c_dev, size_t n_total, size_t tail_len,
                                    uint8_t* proof_out, size_t proof_cap, size_t* proof_len);

/* ---- BLS12-377: the reference's own SIPP instantiation (SURVEY.md §8f-4) ------------------------------------- */
/* `SIPP<Bls12_377, Blake2s>` (sipp/src/lib.rs:228-254, sipp/examples/scaling-ipp.rs:10) on the second parameter set
 * (csrc/bls377.cuh: Fq2 non-residue -5, xi = u, D-type twist, x > 0; ark-ec's default little-endian point
 * serialisation in the Fiat-Shamir seed).  Same conventions as the BLS12-381 entry points: host pointers, Montgomery
 * limbs (12 x 32 bits for the 377-bit Fq, 8 x 32 for the 253-bit Fr), affine points packed x | y (G1 96 B, G2 192 B,
 * identity = all zero), GT = 576 B in arkworks' tower order; proof = log2(n) pairs (z_l, z_r), serialize_uncompressed.
 * One thread per pairing / element: the correctness port of the curve (bit-exact against oracle/bls12_377.py); the
 * lane-role throughput engines are specialised on BLS12-381. */
int ripp377_pairing_ip_affine(ripp_ctx* ctx, const void* g1_aff, size_t n_left, const void* g2_aff, size_t n_right,
                              void* gt_out);
int ripp377_sipp_product_with_coeffs(ripp_ctx* ctx, const void* a_aff, const void* b_aff, const void* r, size_t n,
                                     void* gt_out);
int ripp377_sipp_prove(ripp_ctx* ctx, const void* a_aff, const void* b_aff, const void* r, size_t n, const void* value_gt,
                       uint8_t* proof_out, size_t proof_cap, size_t* proof_len);
int ripp377_sipp_verify(ripp_ctx* ctx, const void* a_aff, const void* b_aff, const void* r, size_t n, const void* value_gt,
                        const uint8_t* proof, size_t proof_len, int* accept);

/* ---- verifiers (SURVEY.md §8 rows a13, a17, a20, a22) ----------------------------------------- */
/* All arithmetic of the verifiers runs on the GPU (GT multi-exponentiation, MSMs, pairings); the host
 * recomputes the Fiat-Shamir chain from the proof bytes.  Inputs are arkworks serialize_uncompressed
 * bytes as the provers above emit them.  *accept = 1 / 0 is the reference's Ok(true) / Ok(false);
 * bytes that do not decode (non-canonical field element, point off the curve, wrong length) fail with
 * RIPP_ERR_ARG, as ark-serialize would before the reference's verify is ever called.
 *
 * `com`: the statement, serialised commitment by commitment --
 *     com_a || com_b || com_t          (com_t = IdentityOutput: u64 LE length 1, then the value)
 *     com_a || com_t                   for the *_SSM kinds (the right commitment is the placeholder). */

/* prod_i g_i^(s_i) in GT, device pointers (g: n x 576 B, s: n Fr Montgomery): `PairingOutput * Fr`
 * (mul_helper with T = GT, ip_proofs/src/lib.rs:15-19), the primitive of gipa.rs:355-357 and
 * sipp/src/lib.rs:152-160.  Generic Fq12 squarings: inputs need not lie in the cyclotomic subgroup. */
int ripp_gt_multiexp_dev(ripp_ctx* ctx, const void* gt_dev, const void* fr_dev, size_t n, void* gt_out_dev);

/* GIPA::verify (gipa.rs:135-160: _compute_recursive_challenges :322-363, _compute_final_commitment_keys
 * :365-399 as one MSM per key vector, _verify_base_commitment :401-415); for the *_SSM kinds
 * GIPAWithSSM::verify_with_structured_scalar_message (structured_scalar_message.rs:86-127) with
 * scalar_b = one Fr (host, Montgomery), w_dev NULL.  v_dev / w_dev: the n commitment keys (device, affine). */
int ripp_gipa_verify_dev(ripp_ctx* ctx, int kind, const void* v_dev, const void* w_dev, size_t n, const uint8_t* com,
                         size_t com_len, const void* scalar_b, const uint8_t* proof, size_t proof_len, int* accept);

/* VerifierSRS (tipa/mod.rs:88-94), host, Montgomery affine, packed: g (96 B) | h (192 B) | g_beta (96 B) |
 * h_alpha (192 B).
 * TIPA::verify_with_srs_shift (tipa/mod.rs:242-301; `shift` = r_shift, NULL for TIPA::verify) for kinds with a
 * G1 right key; TIPAWithSSM::verify_with_structured_scalar_message (structured_scalar_message.rs:270-331;
 * `shift` = scalar_b, required) for the *_SSM kinds.  The KZG checks are verify_commitment_key_g{1,2}_kzg_opening
 * (tipa/mod.rs:340-370). */
int ripp_tipa_verify(ripp_ctx* ctx, int kind, const void* vsrs, const uint8_t* com, size_t com_len, const void* shift,
                     const uint8_t* proof, size_t proof_len, int* accept);

/* verify_aggregate_proof (applications/groth16_aggregation.rs:162-231).
 * vk (ark-groth16 VerifyingKey), host, Montgomery affine, packed: alpha_g1 (96 B) | beta_g2 (192 B) |
 * gamma_g2 (192 B) | delta_g2 (192 B) | gamma_abc_g1[m + 1] (96 B each); public_inputs: n x m Fr (host,
 * Montgomery, row = one proof's inputs); proof: the bytes ripp_tipp_aggregate emits. */
int ripp_tipp_verify_aggregate(ripp_ctx* ctx, const void* vsrs, const void* vk, size_t m, const void* public_inputs,
                               size_t n, const uint8_t* proof, size_t proof_len, int* accept);

/* verify_aggregate_proof for `count` aggregates under one VerifierSRS and one VerifyingKey, one status per aggregate.
 * status_out[k] is what ripp_tipp_verify_aggregate reports for aggregate k alone: */
typedef enum ripp_agg_status {
  RIPP_AGG_OK = 0,              /* accepted */
  RIPP_AGG_MALFORMED = 1,       /* the bytes do not decode (length, non-canonical field element, off the curve) */
  RIPP_AGG_NOT_IN_SUBGROUP = 2, /* a G1 / G2 / GT element outside the prime-order subgroup */
  RIPP_AGG_REJECTED = 3         /* decodes, verify_aggregate_proof returns false */
} ripp_agg_status;
/* vsrs, vk, m: as ripp_tipp_verify_aggregate, shared by all aggregates.  n[k]: aggregate k's number of Groth16
 * proofs (may differ between aggregates).  public_inputs: the rows of all aggregates back to back, sum_k n[k] rows of
 * m Fr (host, Montgomery).  proofs: the AggregateProof bytes back to back, proof_lens[k] bytes for aggregate k,
 * proofs_len in all.  *n_accepted counts the RIPP_AGG_OK.  A bad aggregate is data, not an error: the call fails
 * with RIPP_ERR_ARG only for null pointers, n[k] == 0, m outside 1..1024, proof_lens that do not sum to proofs_len
 * and count > 2^24; count == 0 returns RIPP_OK.  Deterministic (no randomness), and no status depends on the other
 * members.  The kernel launches do not grow with count (subgroup checks, one G1 scaling, segmented sums, the GT folds,
 * one Miller and one final-exponentiation launch for all aggregates: DESIGN.md §4); two host synchronisations. */
int ripp_tipp_verify_aggregate_batch(ripp_ctx* ctx, const void* vsrs, const void* vk, size_t m, size_t count,
                                     const size_t* n, const void* public_inputs, const uint8_t* proofs,
                                     size_t proofs_len, const size_t* proof_lens, uint8_t* status_out,
                                     size_t* n_accepted);

/* SIPP::verify (sipp/src/lib.rs:109-180): inputs as ripp_sipp_prove, proof = its output. */
int ripp_sipp_verify(ripp_ctx* ctx, const void* a_aff, const void* b_aff, const void* r, size_t n, const void* value_gt,
                     const uint8_t* proof, size_t proof_len, int* accept);

/* ---- polynomial commitments (ip_proofs/src/applications/poly_commit/{mod,transparent}.rs; BLS12-381) ---------------- */
/* Coefficient layout.  A bivariate polynomial is ONE device array of `len` Fr (Montgomery), read row-major with row
 * length m = y_degree + 1: coefficient j of Y polynomial i sits at i * m + j, and everything at or beyond `len` is zero.
 * With n = x_degree + 1 rows, len <= n * m.  A univariate polynomial of degree < n * m is already in this layout: it is
 * the bivariate form UnivariatePolynomialCommitment builds (mod.rs:286-377), opened at (z^m, z), so the univariate and
 * transparent-univariate wrappers map degrees and the point only.  Ragged Y polynomials are padded to m by the caller.
 * n and m must be powers of two (RIPP_ERR_NOT_POW2); n <= 2^16, n * m <= 2^24 (the segmented MSM's limits), null
 * pointers and len > n * m give RIPP_ERR_ARG.  The limits cover univariate degree 2^24 - 1, i.e. (255, 65535). */
typedef enum ripp_pc_kind {
  RIPP_PC_TRUSTED = 0,    /* BivariatePolynomialCommitment (mod.rs:153-284): KZG first tier, TIPAWithSSM second tier */
  RIPP_PC_TRANSPARENT = 1 /* TransparentBivariatePolynomialCommitment (transparent.rs:85-213): Pedersen<G1> first tier,
                             GIPA with structured scalar message on both tiers */
} ripp_pc_kind;

/* Division by (X - z): q = (f - f(z)) / (X - z) (len - 1 Fr, q_out_dev; may be NULL when len <= 1) and the remainder
 * f(z) (one Fr, eval_out_dev, may be NULL), the synthetic division of KZG::open (mod.rs:98-104) as a parallel scan of
 * its linear recurrence.  coeffs_dev: len Fr, lowest degree first; z_host: one Fr (host).  q must not overlap coeffs.
 * len = 0 gives f(z) = 0.  Asynchronous on the context's stream. */
int ripp_fr_div_linear_dev(ripp_ctx* ctx, const void* coeffs_dev, size_t len, const void* z_host, void* q_out_dev,
                           void* eval_out_dev);
/* KZG::commit (mod.rs:85): sum_i coeffs[i] powers[i] over the first len of n_powers G1 powers g^(alpha^i) (device);
 * len > n_powers: RIPP_ERR_ARG; len = 0: the identity.  One affine point to device memory, asynchronous. */
int ripp_pc_kzg_commit_dev(ripp_ctx* ctx, const void* powers_dev, size_t n_powers, const void* coeffs_dev, size_t len,
                           void* g1_aff_out_dev);
/* KZG::open (mod.rs:98-104) at z_host: the quotient on the device, then one MSM.  eval_out_dev (nullable) receives
 * f(z).  len <= 1 has an empty quotient: the proof is the identity.  Asynchronous. */
int ripp_pc_kzg_open_dev(ripp_ctx* ctx, const void* powers_dev, size_t n_powers, const void* coeffs_dev, size_t len,
                         const void* z_host, void* g1_aff_out_dev, void* eval_out_dev);
/* KZG::verify (mod.rs:120-130) as one two-pair product e(com - g eval, h) e(-proof, h_alpha - h z) == 1.  vsrs: the
 * VerifierSRS layout of ripp_tipa_verify; com, proof: G1 affine (host, Montgomery); z, eval: Fr (host). */
int ripp_pc_kzg_verify(ripp_ctx* ctx, const void* vsrs, const void* com, const void* z, const void* eval, const void* proof,
                       int* accept);

/* Commit (mod.rs:186 / transparent.rs:106-119): the n first-tier commitments of the Y polynomials over the m shared
 * first-tier bases (trusted: the KZG powers g^(alpha^j); transparent: the Pedersen key) as ONE segmented MSM
 * (y_coms_dev: n G1 affine, device), then the AFGHO pairing product with the n second-tier G2 keys (trusted: the even
 * powers h^(beta^(2i)); transparent: the second-tier key).  gt_out: the commitment (576 B, host).  Synchronous.  Apart
 * from the pairing product's reduction tree (log n depth), the number of kernel launches does not depend on n. */
int ripp_pc_commit_dev(ripp_ctx* ctx, const void* first_tier_dev, size_t m, const void* second_tier_dev, size_t n,
                       const void* coeffs_dev, size_t len, void* gt_out, void* y_coms_dev);
/* Open at (x, y) (host Fr).  trusted (mod.rs:211-241 and on): srs_g2_dev = h_beta_powers (2 n - 1 G2), the argument is
 * TIPAWithSSM over (y_coms, powers of x) and the KZG opening of y_eval at y; transparent (transparent.rs:137 and on):
 * srs_g2_dev unused, GIPA MULTIEXP_SSM over (y_coms, powers of x) and GIPA SCALAR_SSM_G1 over (y_eval, powers of y).
 * Powers, the row combination y_eval, y_eval_comm and the quotient stay on the device.  proof_out: the OpeningProof
 * bytes (trusted: ip_proof || y_eval_comm || kzg_proof; transparent: second_tier_ip_proof || y_eval_comm ||
 * first_tier_ip_proof); eval_out (host, nullable): f(x, y).  The trusted opening needs n >= 2 (a TIPA of one element
 * has no challenge for its KZG opening; the reference panics at tipa/mod.rs:199): n = 1 gives RIPP_ERR_ARG before any
 * work is launched.  Synchronous. */
int ripp_pc_open_dev(ripp_ctx* ctx, int kind, const void* first_tier_dev, size_t m, const void* second_tier_dev, size_t n,
                     const void* srs_g2_dev, const void* coeffs_dev, size_t len, const void* y_coms_dev, const void* x_host,
                     const void* y_host, uint8_t* proof_out, size_t proof_cap, size_t* proof_len, void* eval_out);
/* Verify an opening of com_gt (host GT, as ripp_pc_commit_dev returns it) at (x, y) to eval (host Fr).  trusted
 * (BivariatePolynomialCommitment::verify): vsrs only (keys and n, m unused), ripp_tipa_verify on com || IdentityOutput(y_eval_comm) plus the
 * KZG check; transparent (the transparent verify): first / second-tier keys with m, n, two ripp_gipa_verify_dev.
 * Undecodable bytes: RIPP_ERR_ARG. */
int ripp_pc_verify(ripp_ctx* ctx, int kind, const void* vsrs, const void* first_tier_dev, size_t m, const void* second_tier_dev,
                   size_t n, const void* com_gt, const void* x_host, const void* y_host, const void* eval, const uint8_t* proof,
                   size_t proof_len, int* accept);

/* ---- diagnostics --------------------------------------------------------------------------- */
/* Element-wise primitive ops on device, used by the GPU parity tests to pin the PTX limb layer:
 * op in ripp_test_op; a, b, r are HOST arrays of n elements of the op's operand size. */
typedef enum ripp_test_op {
  RIPP_OP_FQ_MUL = 0, RIPP_OP_FQ_ADD, RIPP_OP_FQ_SUB, RIPP_OP_FQ_INV, RIPP_OP_FQ_HALF,
  RIPP_OP_FR_MUL, RIPP_OP_FR_ADD, RIPP_OP_FR_SUB, RIPP_OP_FR_INV,
  RIPP_OP_FQ2_MUL, RIPP_OP_FQ2_SQR, RIPP_OP_FQ2_INV,
  RIPP_OP_FQ12_MUL, RIPP_OP_FQ12_SQR, RIPP_OP_FQ12_INV, RIPP_OP_FQ12_CYC_SQR, RIPP_OP_FQ12_FROB1,
  RIPP_OP_FINAL_EXP, RIPP_OP_MILLER,       /* MILLER: a = G1 affine, b = G2 affine, r = Fq12 */
  RIPP_OP_G1_ADD, RIPP_OP_G1_DBL, RIPP_OP_G2_ADD, RIPP_OP_G2_DBL /* affine in, affine out */
} ripp_test_op;
int ripp_test_elementwise(ripp_ctx* ctx, int op, const void* a, const void* b, void* r, size_t n);

/* Integer-pipe microbenchmark that defines the roofline denominator (SURVEY.md §8d):
 * kind 0 = independent IMAD.WIDE.U32 chains (one MAC32 each), 1 = 32-bit IMAD chains,
 * 2 = carry-chained mad.lo.cc/madc.hi.cc pairs.  Returns multiply-accumulates per second
 * and the average kernel time in ms. */
int ripp_bench_imad(ripp_ctx* ctx, int kind, int iters, double* macs_per_s, double* ms);

#ifdef __cplusplus
}
#endif
#endif /* RIPP_B200_H */
