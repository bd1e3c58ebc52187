"""The oracle of Groth16 verification by random linear combination (oracle/groth16_rlc.py): ChaCha20 scalars with
known answers, per-segment normalisation, and the segment check in exponent space and over the pairing against the
per-proof verdicts (oracle/groth16.py)."""
import random

import pytest

from oracle import bls12_381 as E
from oracle import encoding as enc
from oracle import groth16 as G
from oracle import groth16_rlc as Q
from oracle import synth as OS

SEED = bytes(range(32))


def test_scalars_are_chacha20_keystream_chunks():
    # RFC 8439 A.1 test vector 1 (key 0, counter 0, nonce 0): the keystream starts 76 b8 e0 ad a0 f1 3d 90 ...
    r = Q.rlc_scalars(bytes(32), [True] * 9, 100)
    assert r[0] == int.from_bytes(bytes.fromhex("76b8e0ada0f13d90405d6ae55386bd28"), "little")
    assert r[1] == int.from_bytes(bytes.fromhex("bdd219b8a08ded1aa836efcc8b770dc7"), "little")
    ks = enc.chacha20_block(SEED, 0) + enc.chacha20_block(SEED, 1) + enc.chacha20_block(SEED, 2)
    r = Q.rlc_scalars(SEED, [True] * 12, 100)
    assert r[:11] == [int.from_bytes(ks[16 * i : 16 * i + 16], "little") for i in range(11)]
    assert all(v < 1 << 128 for v in r[:11])


@pytest.mark.parametrize("s", [1, 3, 7, 58, 200])
def test_members_of_each_segment_sum_to_one(s):
    rng = random.Random(s)
    members = [rng.random() < 0.8 for _ in range(61)]
    members[7 : 7 + min(s, 5)] = [False] * min(s, 5)
    r = Q.rlc_scalars(SEED, members, s)
    assert all(v == 0 for v, mem in zip(r, members) if not mem)
    for lo in range(0, len(members), s):
        idx = [i for i in range(lo, min(len(members), lo + s)) if members[i]]
        if idx:
            assert sum(r[i] for i in idx) % E.R == 1
            assert r[idx[0]] < 1 << 128 or len(idx) == 1
    # a one-member segment has r = 1
    assert Q.rlc_scalars(SEED, [True] * 5, 1) == [1] * 5


def _batch(n, m, seed=3):
    sc, proofs, inputs = OS.groth16_instance_scalars(n, m, seed)
    return sc["vk"], sc["ic"], list(proofs), [list(x) for x in inputs]


@pytest.mark.parametrize("kind", G.GROTH16_TAMPER)
def test_every_tamper_class_fails_its_segment(kind):
    vk, ic, proofs, inputs = _batch(9, 2)
    G.groth16_tamper(vk, ic, proofs, inputs, kind, 4, 5 if kind == "b_swapped" else None)
    r = Q.rlc_scalars(SEED, [True] * 9, 9)
    assert not Q.rlc_segment_exponent(vk, ic, proofs, inputs, r, list(range(9)))
    # the other segments of a split batch still pass
    r = Q.rlc_scalars(SEED, [True] * 9, 3)
    assert [Q.rlc_segment_exponent(vk, ic, proofs, inputs, r, list(range(lo, lo + 3))) for lo in (0, 3, 6)] == [True, False, True]


def test_equal_errors_are_caught():
    vk, ic, proofs, inputs = _batch(6, 1)
    for i in range(6):
        G.groth16_tamper(vk, ic, proofs, inputs, "c_plus_g", i)
    r = Q.rlc_scalars(SEED, [True] * 6, 6)
    assert not Q.rlc_segment_exponent(vk, ic, proofs, inputs, r, list(range(6)))


@pytest.mark.parametrize("m", [0, 1, 5])
def test_valid_and_edge_segments_pass_and_one_member_is_the_per_proof_check(m):
    vk, ic, proofs, inputs, kinds = G.groth16_mixed_scalars(m)
    truth = [G.groth16_exponent_verdict(vk, ic, p, x) for p, x in zip(proofs, inputs)]
    valid = [i for i, t in enumerate(truth) if t]
    assert any(kinds[i] in G.GROTH16_EDGE for i in valid)
    r = Q.rlc_scalars(SEED, truth, len(proofs))
    assert Q.rlc_segment_exponent(vk, ic, proofs, inputs, r, valid)
    r = Q.rlc_scalars(SEED, [True] * len(proofs), 1)
    assert [Q.rlc_segment_exponent(vk, ic, proofs, inputs, r, [i]) for i in range(len(proofs))] == truth


@pytest.mark.parametrize("s", [1, 7, 58])
def test_expected_verdicts_equal_the_per_proof_verdicts(s):
    vk, ic, proofs, inputs, kinds = G.groth16_mixed_scalars(1)
    truth = [G.groth16_exponent_verdict(vk, ic, p, x) for p, x in zip(proofs, inputs)]
    n = len(proofs)
    got, nre = Q.rlc_expected(SEED, [True] * n, s, lambda r, idx: Q.rlc_segment_exponent(vk, ic, proofs, inputs, r, idx), truth)
    assert got == truth
    failing = {i // s for i, t in enumerate(truth) if not t}
    assert nre == sum(min(n, (k + 1) * s) - k * s for k in failing)


def test_pairing_check_equals_exponent_check():
    vk, ic, proofs, inputs, kinds = G.groth16_mixed_scalars(1)
    pick = [0, 1, kinds.index("p_identity"), kinds.index("c_identity")]  # valid, C + G, and two valid edge cases
    sub = [proofs[i] for i in pick]
    xs = [inputs[i] for i in pick]
    vkp, pts = G.groth16_points(vk, ic, sub)
    pvk = G.prepare_verifying_key(vkp)
    for members, want in (([True, False, True, True], True), ([True] * 4, False)):
        r = Q.rlc_scalars(SEED, members, 4)
        idx = [i for i in range(4) if members[i]]
        assert Q.rlc_segment_exponent(vk, ic, sub, xs, r, idx) == want
        assert Q.rlc_segment_check(pvk, pts, xs, r, idx) == want
