"""ORACLE (test infrastructure, NOT product code) -- encodings for the decoders' tests: a deterministic mixed batch
covering every status of oracle/serde.py's de_g1 / de_g2 in either mode, the named malformed cases whose arkworks
verdicts tools/ark_golden dumps, and proof records (ark-groth16 `Proof { a, b, c }`) from packed Montgomery words."""
import numpy as np

from . import bls12_381 as E
from . import serde as S
from . import synth as OS

P = E.P
_RQ_INV = pow(1 << 384, -1, P)


def _patch(b, first=None, xor_first=0):
    b = bytearray(b)
    if first is not None:
        b[0] = first
    b[0] ^= xor_first
    return bytes(b)


def _fq_be(v, flags=0):
    b = bytearray(v.to_bytes(48, "big"))
    b[0] |= flags
    return bytes(b)


def _no_sqrt_x(group, seed):
    """An x for which x^3 + b has no square root."""
    i = 0
    while True:
        if group == 1:
            x = OS.scalar("serde-nosqrt", i, seed) % P
            if OS._fp_sqrt((x**3 + 4) % P) is None:
                return x
        else:
            x = (OS.scalar("serde-nosqrt", i, seed) % P, OS.scalar("serde-nosqrt'", i, seed) % P)
            if OS._fp2_sqrt(E.f2_add(E.f2_mul(E.f2_sqr(x), x), E.B2)) is None:
                return x
        i += 1


def named_cases(group, compressed, seed=0):
    """[(name, bytes)]: one encoding per rejection rule plus valid ones (P, -P, the identity, the generator)."""
    ser = (S.ser_g1_compressed if compressed else S.ser_g1) if group == 1 else (S.ser_g2_compressed if compressed else S.ser_g2)
    mul, gen, neg = (E.g1_mul, E.G1_GEN, E.g1_neg) if group == 1 else (E.g2_mul, E.G2_GEN, E.g2_neg)
    p = mul(gen, OS.scalar("serde-p", 0, seed))
    good = ser(p)
    size = len(good)
    cases = [("valid", good), ("valid_neg", ser(neg(p))), ("identity", ser(None)), ("generator", ser(gen))]
    c = 0x80 if compressed else 0
    # flags
    cases.append(("flag_wrong_mode", _patch(good, xor_first=0x80)))
    if compressed:
        cases.append(("flag_sort_with_infinity", _patch(ser(None), xor_first=0x20)))
    else:
        cases.append(("flag_sort_uncompressed", _patch(good, xor_first=0x20)))
    cases.append(("flag_infinity_nonzero_x", _patch(good, first=(good[0] & 0x1F) | 0x40 | c)))
    cases.append(("flag_infinity_nonzero_last", bytes([0x40 | c]) + bytes(size - 2) + b"\x01"))
    # non-canonical: x = p, and the last coordinate = p (uncompressed y / compressed G2 x.c0)
    cases.append(("x_eq_p", _fq_be(P, c) + good[48:]))
    cases.append(("last_eq_p", good[: size - 48] + _fq_be(P, c if size == 48 else 0)))
    cases.append(("x_max", bytes([0x1F | c]) + b"\xff" * 47 + good[48:]))
    # off the curve
    if compressed:
        cases.append(("x_no_sqrt", _x_only(group, _no_sqrt_x(group, seed))))
    else:
        y = p[1] + 1 if group == 1 else (p[1][0], (p[1][1] + 1) % P)
        cases.append(("y_off_curve", ser((p[0], y % P if group == 1 else y))))
    # on the curve, outside the prime-order subgroup
    off = OS.g1_point_off_subgroup(seed) if group == 1 else OS.g2_point_off_subgroup(seed)
    cases.append(("off_subgroup", ser(off)))
    return cases


def _x_only(group, x):
    if group == 1:
        return _fq_be(x, 0x80)
    return _fq_be(x[1], 0x80) + _fq_be(x[0])


def mixed_batch(group, compressed, count, seed=0):
    """`count` encodings cycling through every kind of named_cases with fresh points, plus random bytes with valid-looking
    flags.  Deterministic in (group, compressed, count, seed)."""
    out = []
    k = 0
    while len(out) < count:
        for _, b in named_cases(group, compressed, seed + k):
            out.append(b)
        junk = bytearray(OS.blake2b(b"serde-junk" + bytes([group, compressed]) + k.to_bytes(8, "little")))
        junk = (junk * 4)[: 48 * (1 if compressed else 2) * (1 if group == 1 else 2)]
        junk[0] = (junk[0] & 0x1F) | (0x80 if compressed else 0)
        out.append(bytes(junk))
        k += 1
    return out[:count]


# ---- ark-groth16 Proof records from packed Montgomery words (codec / ripp_b200 layout) --------------------------
def _fq_canon(words):
    return int.from_bytes(np.ascontiguousarray(words, dtype=np.uint32).tobytes(), "little") * _RQ_INV % P


def g1_words_to_bytes(w, compressed):
    w = np.asarray(w)
    if not w.any():
        return S.ser_g1_compressed(None) if compressed else S.ser_g1(None)
    pt = (_fq_canon(w[:12]), _fq_canon(w[12:24]))
    return S.ser_g1_compressed(pt) if compressed else S.ser_g1(pt)


def g2_words_to_bytes(w, compressed):
    w = np.asarray(w)
    if not w.any():
        return S.ser_g2_compressed(None) if compressed else S.ser_g2(None)
    pt = ((_fq_canon(w[:12]), _fq_canon(w[12:24])), (_fq_canon(w[24:36]), _fq_canon(w[36:48])))
    return S.ser_g2_compressed(pt) if compressed else S.ser_g2(pt)


def proof_records(a_words, b_words, c_words, compressed):
    """n packed G1 / G2 / G1 affine points ((n, 24), (n, 48), (n, 24) uint32) -> n Proof records back to back."""
    a, b, c = (np.asarray(x) for x in (a_words, b_words, c_words))
    return b"".join(g1_words_to_bytes(a[i], compressed) + g2_words_to_bytes(b[i], compressed) + g1_words_to_bytes(c[i], compressed)
                    for i in range(a.shape[0]))


def proof_records_from_points(proofs, compressed):
    """[(A, B, C)] affine tuples -> Proof records."""
    s1 = S.ser_g1_compressed if compressed else S.ser_g1
    s2 = S.ser_g2_compressed if compressed else S.ser_g2
    return b"".join(s1(a) + s2(b) + s1(c) for a, b, c in proofs)
