"""PairingInnerProduct / AFGHO16 commitments on the GPU through the C ABI, against the oracle
(small n, bit-exact) and through size-independent identities at BASELINE.json's sizes.
Mirrors the reference's own tests: dh_commitments/src/afgho16/mod.rs:62-93 (correct message
verifies, wrong message does not, wrong length errors)."""
import random

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import protocols as O
from oracle import synth as OS
from ripp_b200 import _lib, codec as C, synth

pytestmark = pytest.mark.gpu
rnd = random.Random(11)


@pytest.mark.parametrize("n", [0, 1, 2, 31, 33, 64, 100])
def test_pairing_ip_matches_oracle(ctx, n):
    ps, qs = OS.g1_points("t-a", n, seed=n), OS.g2_points("t-b", n, seed=n)
    if n >= 31:  # identities in either slot contribute 1 (SURVEY.md App. A-6)
        ps[3], qs[7] = None, None
    want = E.multi_pairing(ps, qs)
    got = ctx.pairing_ip_affine(C.g1_vec_enc(ps).reshape(n, 24), C.g2_vec_enc(qs).reshape(n, 48))
    assert C.gt_dec(got) == want


def test_pairing_ip_jacobian_inputs(ctx):
    """arkworks `Projective` inputs with arbitrary Z are normalised on the device (lib.rs:80-81)."""
    n = 9
    ps, qs = OS.g1_points("t-a", n, seed=3), OS.g2_points("t-b", n, seed=3)
    g1 = np.stack([C.g1_jac_enc(p, rnd.randrange(1, E.P)) for p in ps[:-1]] + [C.g1_jac_enc(None)])
    g2 = []
    for q in qs:
        z = (rnd.randrange(1, E.P), rnd.randrange(E.P))
        z2 = E.f2_sqr(z)
        g2.append(np.concatenate([C.fq2_enc(E.f2_mul(q[0], z2)), C.fq2_enc(E.f2_mul(q[1], E.f2_mul(z2, z))), C.fq2_enc(z)]))
    got = ctx.pairing_ip(g1, np.stack(g2))
    assert C.gt_dec(got) == E.multi_pairing(ps[:-1] + [None], qs)


def test_length_mismatch_is_an_error(ctx):
    g1, g2 = np.zeros((4, 36), dtype=np.uint32), np.zeros((5, 72), dtype=np.uint32)
    with pytest.raises(_lib.LengthMismatch) as e:
        ctx.pairing_ip(g1, g2)
    assert "4, 5" in str(e.value)


def test_afgho_commitments(ctx):
    """afgho16/mod.rs:62-93 on the mirrored classes."""
    from ripp_b200.dh_commitments import AFGHOCommitmentG1, AFGHOCommitmentG2

    n = 8
    ck = OS.g2_points("ck", n)
    msg = OS.g1_points("msg", n)
    wrong = OS.g1_points("wrong", n)
    com = AFGHOCommitmentG1.commit(ck, msg)
    assert com == O.AFGHOCommitmentG1.commit(ck, msg)
    assert AFGHOCommitmentG1.verify(ck, msg, com)
    assert not AFGHOCommitmentG1.verify(ck, wrong, com)
    with pytest.raises(_lib.LengthMismatch):
        AFGHOCommitmentG1.verify(ck[:-1], msg, com)
    ck1 = OS.g1_points("ck1", n)
    msg2 = OS.g2_points("msg2", n)
    com2 = AFGHOCommitmentG2.commit(ck1, msg2)
    assert com2 == O.AFGHOCommitmentG2.commit(ck1, msg2)
    assert AFGHOCommitmentG2.verify(ck1, msg2, com2)
    assert not AFGHOCommitmentG2.verify(ck1, OS.g2_points("wrong2", n), com2)


@pytest.mark.parametrize("logn", [10, 14])
def test_pairing_ip_bilinearity_at_scale(ctx, logn):
    """prod e(s_i G1, t_i G2) = e(G1, G2)^(sum s_i t_i): checks the full-size device path with one
    oracle pairing.  Points are generated on the GPU and spot-checked against the oracle."""
    n = 1 << logn
    s, t = synth.scalars("big-a", n), synth.scalars("big-b", n)
    a, b = synth.g1_points_dev(ctx, "big-a", n), synth.g2_points_dev(ctx, "big-b", n)
    out = ctx.alloc(576)
    ctx.pairing_ip_dev(a, b, n, out)
    got = C.gt_dec(out.download(144))
    for i in (0, n // 2, n - 1):
        assert C.g1_dec(a.download(24, offset=96 * i)) == E.g1_mul(E.G1_GEN, s[i])
        assert C.g2_dec(b.download(48, offset=192 * i)) == E.g2_mul(E.G2_GEN, t[i])
    e = sum(x * y for x, y in zip(s, t)) % E.R
    assert got == E.gt_pow(E.pairing(E.G1_GEN, E.G2_GEN), e)


def test_sharded_partials_combine(ctx):
    """SURVEY.md §8e: slices -> Miller partials (no final exp) -> combine == whole product; 3 and 9 slices (more than
    eight partials, one of them empty)."""
    n = 96
    a, b = synth.g1_points_dev(ctx, "sh-a", n), synth.g2_points_dev(ctx, "sh-b", n)
    whole = ctx.alloc(576)
    ctx.pairing_ip_dev(a, b, n, whole)
    for cuts in ((0, 40, 41, 96), (0, 1, 10, 20, 20, 33, 50, 64, 80, 96)):
        k = len(cuts) - 1
        parts = ctx.alloc(576 * k)
        for r in range(k):
            lo, hi = cuts[r], cuts[r + 1]
            ctx.miller_partial_dev(a.ptr + 96 * lo, b.ptr + 192 * lo, hi - lo, parts.ptr + 576 * r)
        comb = ctx.alloc(576)
        ctx.gt_combine_dev(parts, k, comb)
        assert (comb.download(144) == whole.download(144)).all(), k
