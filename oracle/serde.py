"""ORACLE (test infrastructure, NOT product code) -- ark-serialize point encodings with validation.

PARITY UNPINNED (see oracle/bls12_381.py).  Compressed encoders next to oracle/encoding.py's uncompressed ser_g1 /
ser_g2 (re-exported here), and the validating decoders de_g1 / de_g2 that the GPU decoders (ripp_b200/csrc/serde.cuh)
and the compiled restatement (oracle/cpu/serde_cpu.cpp) are checked against.
"""
from . import bls12_381 as E
from .encoding import ser_g1, ser_g2  # noqa: F401  (uncompressed forms, for callers that need both modes)


def _lex_largest_fq(y):
    return y > (E.P - 1) // 2


def _lex_largest_fq2(y):
    """ark-ff 0.4 orders Fq2 by c1, then c0: y > -y decided by c1 unless c1 = 0."""
    return _lex_largest_fq(y[1]) if y[1] else _lex_largest_fq(y[0])


def ser_g1_compressed(pt):
    """ark-bls12-381 0.4 compressed G1: big-endian x, flags 0x80 | (0x20 if y is the largest root)."""
    if pt is None:
        return b"\xc0" + b"\x00" * 47
    b = bytearray(pt[0].to_bytes(48, "big"))
    b[0] |= 0x80 | (0x20 if _lex_largest_fq(pt[1]) else 0)
    return bytes(b)


def ser_g2_compressed(pt):
    """ark-bls12-381 0.4 compressed G2: big-endian x.c1 || x.c0, flags as G1 with the Fq2 ordering."""
    if pt is None:
        return b"\xc0" + b"\x00" * 95
    (x0, x1), y = pt
    b = bytearray(x1.to_bytes(48, "big") + x0.to_bytes(48, "big"))
    b[0] |= 0x80 | (0x20 if _lex_largest_fq2(y) else 0)
    return bytes(b)


# ---- validated decoding (ark-serialize 0.4 deserialize_{compressed,uncompressed} with Validate::Yes) -------------
# Restatement of ark-bls12-381 0.4 curves/util.rs (EncodingFlags::get_flags, read_g{1,2}_{compressed,uncompressed})
# and of ark-ec's Valid::check for affine points; PARITY UNPINNED: tools/ark_golden dumps arkworks' verdicts on the
# malformed encodings of serde_cases.py for tests/test_golden_serde.py.
#
# Layout: coordinates big-endian, 48 bytes per Fq; G1 = x or x || y, G2 = x.c1 || x.c0 or x.c1 || x.c0 || y.c1 || y.c0.
# Flags: the top three bits of byte 0 -- 0x80 compressed, 0x40 infinity, 0x20 y lexicographically largest.
# Checks in order; an element reports the first that fails (arkworks' error in brackets):
#   FLAGS           the compression bit does not match the mode, or the sort bit is set without compression or
#                   together with infinity [UnexpectedFlags]; or the infinity bit is set while any other coordinate
#                   bit (flags masked) is non-zero [InvalidData]
#   NONCANONICAL    a coordinate, flag bits masked off, is >= p [InvalidData: deserialize_fq]
#   NOT_ON_CURVE    uncompressed: y^2 != x^3 + b (b = 4, resp. 4 (1 + u)); compressed: x^3 + b has no square root
#                   [InvalidData]
#   NOT_IN_SUBGROUP [r] P != O [InvalidData]
# Root selection (get_point_from_x_unchecked): y or -y such that "y > -y" equals the sort bit; Fq compares canonical
# integers, Fq2 compares c1 first and c0 only when c1 is equal (y.c1 > (p-1)/2, or y.c1 = 0 and y.c0 > (p-1)/2).
OK, FLAGS, NONCANONICAL, NOT_ON_CURVE, NOT_IN_SUBGROUP = range(5)
STATUS_NAMES = ("OK", "FLAGS", "NONCANONICAL", "NOT_ON_CURVE", "NOT_IN_SUBGROUP")


def _decode(data, compressed, degree):
    """-> (status, canonical Fq values in serialised order, sort flag) up to the curve checks."""
    data = bytes(data)
    size = 48 * degree * (1 if compressed else 2)
    if len(data) != size:
        raise ValueError("expected %d bytes, got %d" % (size, len(data)))
    c, inf, largest = data[0] & 0x80, data[0] & 0x40, data[0] & 0x20
    body = bytes([data[0] & 0x1F]) + data[1:]
    if bool(c) != bool(compressed) or (largest and (not c or inf)) or (inf and any(body)):
        return FLAGS, None, largest
    if inf:
        return OK, None, largest
    v = [int.from_bytes(body[i : i + 48], "big") for i in range(0, size, 48)]
    if any(x >= E.P for x in v):
        return NONCANONICAL, None, largest
    return None, v, largest


def de_g1(data, compressed):
    """ark-serialize G1Affine::deserialize_{compressed,uncompressed} with validation -> (point or None, status)."""
    from .synth import _fp_sqrt

    st, v, largest = _decode(data, compressed, 1)
    if st is not None:
        return None, st
    x = v[0]
    rhs = (x * x * x + 4) % E.P
    if compressed:
        y = _fp_sqrt(rhs)
        if y is None:
            return None, NOT_ON_CURVE
        if _lex_largest_fq(y) != bool(largest):
            y = -y % E.P
    else:
        y = v[1]
        if y * y % E.P != rhs:
            return None, NOT_ON_CURVE
    if not E.g1_in_subgroup((x, y)):
        return None, NOT_IN_SUBGROUP
    return (x, y), OK


def de_g2(data, compressed):
    """ark-serialize G2Affine::deserialize_{compressed,uncompressed} with validation -> (point or None, status)."""
    from .synth import _fp2_sqrt

    st, v, largest = _decode(data, compressed, 2)
    if st is not None:
        return None, st
    x = (v[1], v[0])
    rhs = E.f2_add(E.f2_mul(E.f2_sqr(x), x), E.B2)
    if compressed:
        y = _fp2_sqrt(rhs)
        if y is None:
            return None, NOT_ON_CURVE
        if _lex_largest_fq2(y) != bool(largest):
            y = E.f2_neg(y)
    else:
        y = (v[3], v[2])
        if E.f2_sqr(y) != rhs:
            return None, NOT_ON_CURVE
    if not E.g2_in_subgroup((x, y)):
        return None, NOT_IN_SUBGROUP
    return (x, y), OK
