"""The oracle's ark-serialize point encoders / validating decoders (oracle/serde.py) and their compiled CPU
restatement (oracle/cpu/serde_cpu.cpp): round trips, every rejection rule in both modes and both groups, and element-by-element
agreement of the two implementations on a mixed batch."""
import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import serde as S
from oracle import serde_cases as SC
from oracle import synth as OS
from ripp_b200 import codec as C

GROUPS = {
    1: (S.ser_g1_compressed, S.ser_g1, S.de_g1, E.g1_mul, E.g1_neg, E.G1_GEN, C.g1_enc),
    2: (S.ser_g2_compressed, S.ser_g2, S.de_g2, E.g2_mul, E.g2_neg, E.G2_GEN, C.g2_enc),
}


@pytest.mark.parametrize("group", [1, 2])
def test_round_trips(group):
    serc, seru, de, mul, neg, gen, _ = GROUPS[group]
    pts = [None, gen, neg(gen)]
    for i in range(6):
        p = mul(gen, OS.scalar("serde-rt", i))
        pts += [p, neg(p)]
    for p in pts:
        for compressed, ser in ((True, serc), (False, seru)):
            b = ser(p)
            assert len(b) == 48 * group * (1 if compressed else 2)
            assert de(b, compressed) == (p, S.OK)
    # the two roots of one x differ exactly in the sort flag
    p = mul(gen, 99)
    a, b = serc(p), serc(neg(p))
    assert a[1:] == b[1:] and (a[0] ^ b[0]) == 0x20


def test_known_encodings():
    """The compressed generators as the Zcash / IETF BLS12-381 encoding writes them."""
    assert S.ser_g1_compressed(E.G1_GEN).hex().startswith("97f1d3a73197d794")
    assert S.ser_g2_compressed(E.G2_GEN).hex().startswith("93e02b6052719f60")
    assert S.ser_g1_compressed(None) == b"\xc0" + bytes(47)
    assert S.ser_g1(None) == b"\x40" + bytes(95)


EXPECT = {
    "valid": S.OK, "valid_neg": S.OK, "identity": S.OK, "generator": S.OK,
    "flag_wrong_mode": S.FLAGS, "flag_sort_with_infinity": S.FLAGS, "flag_sort_uncompressed": S.FLAGS,
    "flag_infinity_nonzero_x": S.FLAGS, "flag_infinity_nonzero_last": S.FLAGS,
    "x_eq_p": S.NONCANONICAL, "last_eq_p": S.NONCANONICAL, "x_max": S.NONCANONICAL,
    "x_no_sqrt": S.NOT_ON_CURVE, "y_off_curve": S.NOT_ON_CURVE, "off_subgroup": S.NOT_IN_SUBGROUP,
}


@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("compressed", [True, False])
def test_rejection_classes(group, compressed):
    de = GROUPS[group][2]
    cases = SC.named_cases(group, compressed)
    for name, b in cases:
        pt, st = de(b, compressed)
        assert st == EXPECT[name], (name, S.STATUS_NAMES[st])
        if st != S.OK:
            assert pt is None
    assert {EXPECT[n] for n, _ in cases} == set(range(5))


def test_uncompressed_sort_bit_rejected():
    """An uncompressed encoding with the sort bit set is refused (get_flags), even on a valid point."""
    b = bytearray(S.ser_g1(E.G1_GEN))
    b[0] |= 0x20
    assert S.de_g1(bytes(b), False) == (None, S.FLAGS)


@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("compressed", [True, False])
def test_cpu_restatement_matches_oracle(group, compressed):
    from oracle.cpu import serde_binding as binding

    de, enc = GROUPS[group][2], GROUPS[group][6]
    batch = SC.mixed_batch(group, compressed, 300)
    size = len(batch[0])
    # strided, as packed proof records are read: each element followed by 16 bytes of padding
    data = b"".join(b + b"\xa5" * 16 for b in batch)
    pts, st = binding.deserialize(group, data, len(batch), size + 16, compressed)
    for i, b in enumerate(batch):
        want_pt, want_st = de(b, compressed)
        assert st[i] == want_st, (i, S.STATUS_NAMES[st[i]], S.STATUS_NAMES[want_st])
        assert np.array_equal(pts[i], enc(want_pt)), i
    assert set(st.tolist()) == set(range(5))
