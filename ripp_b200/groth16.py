"""Groth16 verification on the GPU with one verdict per proof: ark-groth16 0.4 prepare_verifying_key / verify_proof
for batches (include/ripp_b200.h "Groth16 verification").  Screen proofs from untrusted provers before aggregating
them: a false proof makes the whole aggregate fail verify_aggregate_proof, and this names it.

verify_proofs / verify_proofs_serialized run ark-groth16's verify_proof for every proof.  The _rlc forms check random
linear combinations of segments of proofs and re-check only the proofs of failing segments one by one: the same
verdicts except with probability at most 2^-128 per segment, at a fraction of the cost when most proofs are valid."""
import os

import numpy as np

from . import _lib, codec
from .inner_products import default_context
from .ip_proofs import PROOF_RECORD_BYTES, vk_enc

# ripp_groth16_status: 0..4 the decode status of the first bad point (A, B, C), then these two
OK, FLAGS, NONCANONICAL, NOT_ON_CURVE, NOT_IN_SUBGROUP, INPUT_NONCANONICAL, REJECTED = range(7)
STATUS_NAMES = ("OK", "FLAGS", "NONCANONICAL", "NOT_ON_CURVE", "NOT_IN_SUBGROUP", "INPUT_NONCANONICAL", "REJECTED")


class PreparedVerifyingKey:
    """ark-groth16 PreparedVerifyingKey in device memory (e(alpha, beta), -gamma, -delta, IC_0 and fixed-base tables of
    IC_1..IC_m); owns its buffer."""

    def __init__(self, ctx, vk):
        self.ctx = ctx
        self.m = len(vk["gamma_abc_g1"]) - 1
        if self.m < 0:
            raise ValueError("gamma_abc_g1 is empty")
        self.buf = ctx.alloc(ctx.groth16_pvk_bytes(self.m))
        ctx.groth16_prepare_vk_dev(vk_enc(vk), self.m, self.buf)


def prepare_verifying_key(vk, ctx=None):
    """vk: dict(alpha_g1, beta_g2, gamma_g2, delta_g2, gamma_abc_g1) of affine points (trusted)."""
    return PreparedVerifyingKey(ctx or default_context(), vk)


def verify_proofs(pvk, public_inputs, proofs):
    """verify_proof for every (inputs, proof): public_inputs = one list of Fr ints per proof, proofs = [(A, B, C)]
    affine points (trusted: on the curve and in the subgroup).  -> list of bool.  A row whose length is not m raises
    ValueError, as prepare_inputs fails in ark-groth16."""
    ctx, m, n = pvk.ctx, pvk.m, len(proofs)
    _check_rows(pvk, public_inputs, proofs)
    if n == 0:
        return []
    a, b, c, x = _upload(pvk, public_inputs, proofs)
    out = ctx.alloc(n)
    ctx.groth16_verify_batch_dev(pvk.buf, m, x, a, b, c, n, out)
    ctx.sync()
    return [bool(v) for v in out.download(n, dtype=np.uint8)]


def _seed(seed):
    seed = os.urandom(32) if seed is None else bytes(seed)
    if len(seed) != 32:
        raise ValueError("the seed is %d bytes, not 32" % len(seed))
    return seed


def _check_rows(pvk, public_inputs, proofs):
    if len(public_inputs) != len(proofs):
        raise ValueError("%d rows of public inputs for %d proofs" % (len(public_inputs), len(proofs)))
    for i, x in enumerate(public_inputs):
        if len(x) != pvk.m:
            raise ValueError("proof %d: %d public inputs, the key has %d" % (i, len(x), pvk.m))


def _upload(pvk, public_inputs, proofs):
    ctx = pvk.ctx
    a = ctx.to_device(codec.g1_vec_enc([p[0] for p in proofs]))
    b = ctx.to_device(codec.g2_vec_enc([p[1] for p in proofs]))
    c = ctx.to_device(codec.g1_vec_enc([p[2] for p in proofs]))
    x = ctx.to_device(codec.fr_vec_enc([v for row in public_inputs for v in row])) if pvk.m else None
    return a, b, c, x


def verify_proofs_serialized(pvk, inputs_bytes, data, compressed=True):
    """Untrusted bytes: `data` holds ark-groth16 Proof records back to back (serialize_compressed 192 B /
    serialize_uncompressed 384 B each, no length prefix), `inputs_bytes` the m ark-serialize Fr (32 B little-endian) of
    each proof in the same order.  -> np.ndarray of uint8 statuses (OK .. REJECTED above), one per proof."""
    n = len(data) // PROOF_RECORD_BYTES[bool(compressed)]
    st, _ = pvk.ctx.groth16_verify_serialized(pvk.buf, pvk.m, inputs_bytes, data, n, compressed)
    return st


def verify_proofs_rlc(pvk, public_inputs, proofs, seed=None):
    """verify_proofs by random linear combination: -> (list of bool, number of proofs re-checked one by one).  seed: 32
    bytes unknown to the provers until their proofs are fixed, fresh per call; None draws os.urandom(32)."""
    seed = _seed(seed)
    ctx, n = pvk.ctx, len(proofs)
    _check_rows(pvk, public_inputs, proofs)
    if n == 0:
        return [], 0
    a, b, c, x = _upload(pvk, public_inputs, proofs)
    out = ctx.alloc(n)
    nre = ctx.groth16_verify_rlc_dev(pvk.buf, pvk.m, x, a, b, c, n, seed, out)
    return [bool(v) for v in out.download(n, dtype=np.uint8)], nre


def verify_proofs_serialized_rlc(pvk, inputs_bytes, data, compressed=True, seed=None):
    """verify_proofs_serialized by random linear combination: -> (np.ndarray of uint8 statuses, number of proofs
    re-checked one by one).  Proofs with a decode or input status are left out of the combinations; seed as in
    verify_proofs_rlc."""
    n = len(data) // PROOF_RECORD_BYTES[bool(compressed)]
    st, _, nre = pvk.ctx.groth16_verify_rlc_serialized(pvk.buf, pvk.m, inputs_bytes, data, n, compressed, _seed(seed))
    return st, nre
