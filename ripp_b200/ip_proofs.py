"""Host-side mirror of `ip_proofs/src` (GIPA gipa.rs:16-22,97-178; TIPA tipa/mod.rs:32-39,150-231;
TIPAWithSSM structured_scalar_message.rs:130-268; aggregate_proofs groth16_aggregation.rs:77-160)
over the C ABI.  Values are Python ints / affine tuples; proofs are returned as the arkworks
`serialize_uncompressed` bytes the library emits."""
import numpy as np

from . import _lib, codec
from .inner_products import default_context


class InnerProductArgumentError(Exception):
    """ip_proofs/src/lib.rs:22-43."""


_ENC = {"G1": codec.g1_vec_enc, "G2": codec.g2_vec_enc, "Fr": codec.fr_vec_enc, None: None}
_KIND_TYPES = {
    _lib.GIPA_PAIRING: ("G1", "G2", "G2", "G1"),
    _lib.GIPA_MULTIEXP_PEDERSEN: ("G1", "Fr", "G2", "G1"),
    _lib.GIPA_MULTIEXP_SSM: ("G1", "Fr", "G2", None),
    _lib.GIPA_SCALAR_PEDERSEN_G2_G2: ("Fr", "Fr", "G2", "G2"),
    _lib.GIPA_SCALAR_PEDERSEN_G2_G1: ("Fr", "Fr", "G2", "G1"),
    _lib.GIPA_SCALAR_SSM: ("Fr", "Fr", "G2", None),
    _lib.GIPA_SCALAR_SSM_G1: ("Fr", "Fr", "G1", None),
}


def _upload(ctx, kind, vecs):
    out = []
    for t, v in zip(_KIND_TYPES[kind], vecs):
        out.append(None if t is None else ctx.to_device(_ENC[t](v)))
    return out


def _ser_com(com):
    """(com_a, [com_b,] com_t) -> the byte string of include/ripp_b200.h: the last value is framed as IdentityOutput."""
    *heads, com_t = com
    if isinstance(com_t, (list,)):  # already an IdentityOutput-style one-element list
        (com_t,) = com_t
    return b"".join(codec.ser_value(c) for c in heads) + codec.ser_identity_output(codec.ser_value(com_t))


def vsrs_enc(v_srs):
    """VerifierSRS (tipa/mod.rs:88-94) -> packed g | h | g_beta | h_alpha (144 words)."""
    return np.concatenate([codec.g1_enc(v_srs["g"]), codec.g2_enc(v_srs["h"]), codec.g1_enc(v_srs["g_beta"]),
                           codec.g2_enc(v_srs["h_alpha"])])


def vk_enc(vk):
    """ark-groth16 VerifyingKey dict(alpha_g1, beta_g2, gamma_g2, delta_g2, gamma_abc_g1) -> packed words."""
    return np.concatenate([codec.g1_enc(vk["alpha_g1"]), codec.g2_enc(vk["beta_g2"]), codec.g2_enc(vk["gamma_g2"]),
                           codec.g2_enc(vk["delta_g2"])] + [codec.g1_enc(p) for p in vk["gamma_abc_g1"]])


class GIPA:
    """GIPA<IP, LMC, RMC, IPC, Blake2b> for one of the instantiations in include/ripp_b200.h."""

    def __init__(self, kind, ctx=None):
        self.kind, self.ctx = kind, ctx or default_context()

    def prove(self, values, ck, com):
        """gipa.rs:108-133, the checked entry.  values = (m_a, m_b, ip); ck = (ck_a, ck_b or None, _); com = (com_a, com_b,
        com_t) ((com_a, com_t) for the *_SSM kinds).  Raises InnerProductArgumentError("InnerProductInvalid") when the
        inner product or a commitment does not match, MessageLengthInvalid for a length that is not a power of two."""
        m_a, m_b = values[0], values[1]
        n = len(m_a)
        if len(m_b) != n:
            raise _lib.LengthMismatch(_lib.RIPP_ERR_LEN_MISMATCH, "left length, right length: %d, %d" % (n, len(m_b)))
        a, b, v, w = _upload(self.ctx, self.kind, (m_a, m_b, ck[0], ck[1]))
        try:
            return self.ctx.gipa_prove_checked_dev(self.kind, a, b, v, w, n, _ser_com(com))
        except _lib.RippError as e:
            if e.status == _lib.RIPP_ERR_INNER_PRODUCT:
                raise InnerProductArgumentError("InnerProductInvalid") from e
            if e.status == _lib.RIPP_ERR_NOT_POW2:
                raise InnerProductArgumentError(str(e)) from e
            raise

    def prove_with_aux(self, values, ck):
        """gipa.rs:162-178.  values = (m_a, m_b); ck = (ck_a, ck_b or None).  -> (proof bytes, transcript ints, ck_base bytes)"""
        m_a, m_b = values
        n = len(m_a)
        if n == 0 or n & (n - 1) or len(m_b) != n:
            raise InnerProductArgumentError("left length, right length: %d, %d" % (len(m_a), len(m_b)))
        a, b, v, w = _upload(self.ctx, self.kind, (m_a, m_b, ck[0], ck[1]))
        proof, tr, ckb = self.ctx.gipa_prove_dev(self.kind, a, b, v, w, n)
        return proof, codec.fr_vec_dec(tr), ckb

    def verify(self, ck, com, proof, scalar_b=None):
        """gipa.rs:135-160 (ck = (ck_a, ck_b), com = (com_a, com_b, com_t)); for the *_SSM kinds
        structured_scalar_message.rs:86-127 (ck = (ck_a, None), com = (com_a, com_t), scalar_b).
        com_t is the bare inner-product value; the IdentityOutput framing is added here.  -> bool"""
        ck_a, ck_b = ck
        n = len(ck_a)
        _, _, tv, tw = _KIND_TYPES[self.kind]
        if n == 0 or n & (n - 1) or (tw is not None and len(ck_b) != n):
            raise InnerProductArgumentError("left length, right length: %d, %d" % (n, 0 if ck_b is None else len(ck_b)))
        v = self.ctx.to_device(_ENC[tv](ck_a))
        w = None if tw is None else self.ctx.to_device(_ENC[tw](ck_b))
        sb = None if scalar_b is None else codec.fr_enc(scalar_b).copy()
        return self.ctx.gipa_verify_dev(self.kind, v, w, n, _ser_com(com), proof, sb)


class TIPA:
    """TIPA<IP, LMC, RMC, IPC, Bls12_381, Blake2b> / TIPAWithSSM (for the *_SSM kinds)."""

    def __init__(self, kind, ctx=None):
        self.kind, self.ctx = kind, ctx or default_context()

    @staticmethod
    def setup(alpha, beta, size, ctx=None):
        """TIPA::setup (tipa/mod.rs:150-164) for given trapdoors (the reference draws them with Fr::rand; the caller
        does that here).  -> (SRS dict(g_alpha_powers, h_beta_powers: DeviceBuffers of 2 size - 1 points; g_beta,
        h_alpha: affine tuples), v_srs dict(g, h, g_beta, h_alpha))."""
        ctx = ctx or default_context()
        s1, s2, gb, ha = ctx.tipa_setup_dev(codec.fr_enc(alpha).copy(), codec.fr_enc(beta).copy(), size)
        g_beta, h_alpha = codec.g1_dec(gb), codec.g2_dec(ha)
        srs = {"g_alpha_powers": s1, "h_beta_powers": s2, "g_beta": g_beta, "h_alpha": h_alpha, "size": size}
        g = codec.g1_vec_dec(s1.download((1, 24)))[0]  # power 0 of each tower: the generators (tipa/mod.rs:120-127)
        h = codec.g2_vec_dec(s2.download((1, 48)))[0]
        return srs, {"g": g, "h": h, "g_beta": g_beta, "h_alpha": h_alpha}

    def prove_with_srs_shift(self, srs, values, ck, r_shift=1):
        """tipa/mod.rs:176-231.  srs = (g_alpha_powers, h_beta_powers)."""
        m_a, m_b = values
        n = len(m_a)
        if n == 0 or n & (n - 1) or len(m_b) != n:
            raise InnerProductArgumentError("left length, right length: %d, %d" % (len(m_a), len(m_b)))
        a, b, v, w = _upload(self.ctx, self.kind, (m_a, m_b, ck[0], ck[1]))
        s1 = self.ctx.to_device(codec.g1_vec_enc(srs[0]))
        s2 = self.ctx.to_device(codec.g2_vec_enc(srs[1]))
        return self.ctx.tipa_prove_dev(self.kind, s1, s2, a, b, v, w, n, codec.fr_enc(r_shift).copy())

    def prove(self, srs, values, ck):
        return self.prove_with_srs_shift(srs, values, ck, 1)

    def verify_with_srs_shift(self, v_srs, com, proof, r_shift=1):
        """tipa/mod.rs:242-301.  v_srs = dict(g, h, g_beta, h_alpha); com = (com_a, com_b, com_t).  -> bool"""
        return self.ctx.tipa_verify(self.kind, vsrs_enc(v_srs), _ser_com(com), proof, codec.fr_enc(r_shift).copy())

    def verify(self, v_srs, com, proof):
        return self.verify_with_srs_shift(v_srs, com, proof, 1)

    def verify_with_structured_scalar_message(self, v_srs, com, scalar_b, proof):
        """structured_scalar_message.rs:270-331 (the *_SSM kinds).  com = (com_a, com_t).  -> bool"""
        return self.ctx.tipa_verify(self.kind, vsrs_enc(v_srs), _ser_com(com), proof, codec.fr_enc(scalar_b).copy())


def aggregate_proofs(srs, proofs, ctx=None):
    """groth16_aggregation.rs:77-160.  srs = (g_alpha_powers, h_beta_powers); proofs = [(A, B, C)]."""
    ctx = ctx or default_context()
    n = len(proofs)
    a = ctx.to_device(codec.g1_vec_enc([p[0] for p in proofs]))
    b = ctx.to_device(codec.g2_vec_enc([p[1] for p in proofs]))
    c = ctx.to_device(codec.g1_vec_enc([p[2] for p in proofs]))
    s1 = ctx.to_device(codec.g1_vec_enc(srs[0]))
    s2 = ctx.to_device(codec.g2_vec_enc(srs[1]))
    return ctx.tipp_aggregate_dev(s1, s2, a, b, c, n)


PROOF_RECORD_BYTES = {True: 192, False: 384}


def aggregate_proofs_serialized(srs, data, compressed=True, ctx=None):
    """aggregate_proofs (groth16_aggregation.rs:77-160) starting from the proofs' bytes: `data` holds ark-groth16
    `Proof { a, b, c }` records back to back, each written by serialize_compressed (192 B) or serialize_uncompressed
    (384 B), no length prefix.  Every point is decoded and validated on the GPU (flags, canonical coordinates, curve,
    prime-order subgroup) before the aggregation starts; an invalid record raises RippError naming the first bad proof,
    its component and what is wrong with it.  srs = (g_alpha_powers, h_beta_powers).  -> AggregateProof bytes."""
    ctx = ctx or default_context()
    n = len(data) // PROOF_RECORD_BYTES[bool(compressed)]
    s1 = ctx.to_device(codec.g1_vec_enc(srs[0]))
    s2 = ctx.to_device(codec.g2_vec_enc(srs[1]))
    return ctx.tipp_aggregate_serialized(s1, s2, data, n, compressed)


def verify_aggregate_proof(v_srs, vk, public_inputs, proof, ctx=None):
    """groth16_aggregation.rs:162-231.  public_inputs: one list of Fr per proof; proof: aggregate_proofs' bytes.  -> bool"""
    ctx = ctx or default_context()
    n, m = len(public_inputs), len(public_inputs[0])
    assert len(vk["gamma_abc_g1"]) == m + 1  # :214
    inp = np.ascontiguousarray(np.stack([codec.fr_vec_enc(row) for row in public_inputs]).reshape(n, m, 8))
    return ctx.tipp_verify_aggregate(vsrs_enc(v_srs), np.ascontiguousarray(vk_enc(vk)), inp, proof)


def structured_generators_scalar_power(num, g, s, group, ctx=None):
    """tipa/mod.rs:372-391: [g * s^i for i < num] (g: affine tuple or None = the generator; group 1 / 2).  -> list of points"""
    ctx = ctx or default_context()
    out = ctx.alloc(num * (96 if group == 1 else 192))
    base = None if g is None else (codec.g1_enc(g) if group == 1 else codec.g2_enc(g)).copy()
    ctx.structured_generators_dev(group, base, codec.fr_enc(s).copy(), num, out)
    ctx.sync()
    return (codec.g1_vec_dec if group == 1 else codec.g2_vec_dec)(out.download((num, 24 if group == 1 else 48)))
