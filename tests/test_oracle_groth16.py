"""The Groth16 oracle (oracle/groth16.py over the pure-Python pairing) and its cheap exponent-space truth for
trapdoor-simulated proofs, which the large GPU batches are checked against: they agree on every tamper and edge class."""
import os

import pytest

from oracle import bls12_381 as E
from oracle import groth16 as G
from oracle import serde as S
from oracle import synth as OS


def _mixed(m, seed=0):
    vk, ic, proofs, inputs, kinds = G.groth16_mixed_scalars(m, seed)
    vkp, pts = G.groth16_points(vk, ic, proofs)
    return vk, ic, proofs, inputs, kinds, vkp, pts


def test_accepts_valid_rejects_each_tamper_class():
    vk, ic, proofs, inputs, kinds, vkp, pts = _mixed(2)
    pvk = G.prepare_verifying_key(vkp)
    seen = {}
    for k, p, x in zip(kinds, pts, inputs):
        if k in seen and k == "valid":
            continue
        seen[k] = G.verify_proof(pvk, p, x)
    for k in G.GROTH16_TAMPER + ("a_identity", "b_identity"):
        assert seen[k] is False, k
    for k in ("valid", "p_identity", "c_identity", "input_r_minus_1"):
        assert seen[k] is True, k


@pytest.mark.parametrize("m", [0, 1])
def test_exponent_verdict_equals_pairing_verdict(m):
    """Pins the truth the 2^12 and 2^16 GPU batches use: the exponent-space equation decides as the pairings do."""
    vk, ic, proofs, inputs, kinds, vkp, pts = _mixed(m, seed=3)
    pvk = G.prepare_verifying_key(vkp)
    got = [G.verify_proof(pvk, p, x) for p, x in zip(pts, inputs)]
    want = [G.groth16_exponent_verdict(vk, ic, p, x) for p, x in zip(proofs, inputs)]
    assert got == want
    assert True in got and False in got


def test_edge_points_are_identities():
    vk, ic, proofs, inputs, kinds, vkp, pts = _mixed(1)
    pvk = G.prepare_verifying_key(vkp)
    for k, p, x in zip(kinds, pts, inputs):
        if k == "p_identity":
            assert G.prepare_inputs(pvk, x) is None
        if k == "c_identity":
            assert p[2] is None
        if k == "a_identity":
            assert p[0] is None
        if k == "b_identity":
            assert p[1] is None
        if k == "input_r_minus_1":
            assert x[0] == E.R - 1


def test_length_mismatch_raises():
    vk, ic, proofs, inputs, kinds, vkp, pts = _mixed(1)
    pvk = G.prepare_verifying_key(vkp)
    with pytest.raises(ValueError):
        G.verify_proof(pvk, pts[0], inputs[0] + [1])
    with pytest.raises(ValueError):
        G.verify_proof(pvk, pts[0], [])
    with pytest.raises(ValueError):
        G.groth16_exponent_verdict(vk, ic, proofs[0], inputs[0] + [1])


def test_status_of_serialized_records():
    vk, ic, proofs, inputs, kinds, vkp, pts = _mixed(1)
    pvk = G.prepare_verifying_key(vkp)
    i_ok, i_bad = kinds.index("valid"), kinds.index("c_plus_g")

    def rec(p, compressed):
        if compressed:
            return S.ser_g1_compressed(p[0]) + S.ser_g2_compressed(p[1]) + S.ser_g1_compressed(p[2])
        return S.ser_g1(p[0]) + S.ser_g2(p[1]) + S.ser_g1(p[2])

    def xb(x):
        return b"".join(v.to_bytes(32, "little") for v in x)

    for compressed in (True, False):
        assert G.status_serialized(pvk, rec(pts[i_ok], compressed), xb(inputs[i_ok]), compressed) == S.OK
        assert G.status_serialized(pvk, rec(pts[i_bad], compressed), xb(inputs[i_bad]), compressed) == G.REJECTED
        big = xb([inputs[i_ok][0] + E.R])
        assert G.status_serialized(pvk, rec(pts[i_ok], compressed), big, compressed) == G.INPUT_NONCANONICAL
        r = bytearray(rec(pts[i_ok], compressed))
        r[0] ^= 0x80  # A: wrong compression flag, reported before the inputs
        assert G.status_serialized(pvk, bytes(r), big, compressed) == S.FLAGS


def test_golden_case_file_is_current():
    """The committed proofs whose ark-groth16 verdicts tools/ark_golden dumps are the oracle's m = 1 mixed batch."""
    path = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "groth16_cases.txt")
    assert open(path).read() == G.golden_case_lines(), "regenerate tests/golden/groth16_cases.txt from oracle/groth16.py"
