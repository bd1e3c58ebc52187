"""Groth16 verification on the GPU with one verdict per proof: ark-groth16 0.4 prepare_verifying_key / verify_proof
for batches (include/ripp_b200.h "Groth16 verification").  Screen proofs from untrusted provers before aggregating
them: a false proof makes the whole aggregate fail verify_aggregate_proof, and this names it."""
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
    if len(public_inputs) != n:
        raise ValueError("%d rows of public inputs for %d proofs" % (len(public_inputs), n))
    for i, x in enumerate(public_inputs):
        if len(x) != m:
            raise ValueError("proof %d: %d public inputs, the key has %d" % (i, len(x), m))
    if n == 0:
        return []
    a = ctx.to_device(codec.g1_vec_enc([p[0] for p in proofs]))
    b = ctx.to_device(codec.g2_vec_enc([p[1] for p in proofs]))
    c = ctx.to_device(codec.g1_vec_enc([p[2] for p in proofs]))
    x = ctx.to_device(codec.fr_vec_enc([v for row in public_inputs for v in row])) if m else None
    out = ctx.alloc(n)
    ctx.groth16_verify_batch_dev(pvk.buf, m, x, a, b, c, n, out)
    ctx.sync()
    return [bool(v) for v in out.download(n, dtype=np.uint8)]


def verify_proofs_serialized(pvk, inputs_bytes, data, compressed=True):
    """Untrusted bytes: `data` holds ark-groth16 Proof records back to back (serialize_compressed 192 B /
    serialize_uncompressed 384 B each, no length prefix), `inputs_bytes` the m ark-serialize Fr (32 B little-endian) of
    each proof in the same order.  -> np.ndarray of uint8 statuses (OK .. REJECTED above), one per proof."""
    n = len(data) // PROOF_RECORD_BYTES[bool(compressed)]
    st, _ = pvk.ctx.groth16_verify_serialized(pvk.buf, pvk.m, inputs_bytes, data, n, compressed)
    return st
