"""Groth16 verification with one verdict per proof on the GPU (csrc/groth16.cu): verdicts equal the pairing oracle's
(oracle/groth16.py) on mixed batches with every tamper and edge class, statuses of untrusted bytes equal the oracle's,
keys are reusable, 2^12 and 2^16 batches equal the exponent-space truth, and the verdicts tie in with the aggregation."""
import json
import os
import random

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import groth16 as G
from oracle import serde as S
from oracle import serde_cases as SC
from oracle import synth as OS
from ripp_b200 import _lib, codec as C, synth
from ripp_b200 import groth16 as R
from ripp_b200.ip_proofs import vk_enc

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ark_golden.json")


def _mixed(m, seed=0):
    vk, ic, proofs, inputs, kinds = G.groth16_mixed_scalars(m, seed)
    vkp, pts = G.groth16_points(vk, ic, proofs)
    return vkp, pts, inputs, kinds


@pytest.fixture(scope="module")
def mixed():
    out = {}
    for m in (0, 1, 5):
        vkp, pts, inputs, kinds = _mixed(m)
        pvk = G.prepare_verifying_key(vkp)
        out[m] = (vkp, pts, inputs, kinds, [G.verify_proof(pvk, p, x) for p, x in zip(pts, inputs)])
    return out


@pytest.mark.parametrize("m", [0, 1, 5])
def test_verdicts_match_oracle(ctx, mixed, m):
    vkp, pts, inputs, kinds, want = mixed[m]
    assert True in want and False in want
    pvk = R.prepare_verifying_key(vkp, ctx)
    # e(alpha, beta) of the prepared key (eighteen-lane path) is the oracle's; the per-proof values come from the
    # six-lane shape, and valid proofs are accepted only if the two agree
    assert C.gt_dec(pvk.buf.download(144)) == E.pairing(vkp["alpha_g1"], vkp["beta_g2"])
    got = R.verify_proofs(pvk, inputs, pts)
    assert got == want, [(k, g, w) for k, g, w in zip(kinds, got, want) if g != w]
    for n in (1, 2, 37):  # partial groups (five per warp) and warps (four per CTA)
        idx = [(7 * i + 3) % len(pts) for i in range(n)]
        assert R.verify_proofs(pvk, [inputs[i] for i in idx], [pts[i] for i in idx]) == [want[i] for i in idx], n


def test_row_length_mismatch_raises(ctx, mixed):
    vkp, pts, inputs, kinds, want = mixed[1]
    pvk = R.prepare_verifying_key(vkp, ctx)
    with pytest.raises(ValueError):
        R.verify_proofs(pvk, [inputs[0] + [1]], pts[:1])
    with pytest.raises(ValueError):
        R.verify_proofs(pvk, inputs[:2], pts[:1])


def _record(p, compressed):
    if compressed:
        return S.ser_g1_compressed(p[0]) + S.ser_g2_compressed(p[1]) + S.ser_g1_compressed(p[2])
    return S.ser_g1(p[0]) + S.ser_g2(p[1]) + S.ser_g1(p[2])


def _xbytes(rows):
    return b"".join(v.to_bytes(32, "little") for row in rows for v in row)


def _serialized_batch(pts, inputs, compressed, seed=0):
    """Records of the mixed batch with bad encodings (oracle/serde_cases.py) put into A, B or C of some proofs and
    non-canonical inputs into others."""
    rng = random.Random(seed)
    recs = [bytearray(_record(p, compressed)) for p in pts]
    rows = [list(x) for x in inputs]
    g1b = 48 if compressed else 96
    bad1 = [b for name, b in SC.named_cases(1, compressed, seed) if not name.startswith(("valid", "identity", "generator"))]
    bad2 = [b for name, b in SC.named_cases(2, compressed, seed) if not name.startswith(("valid", "identity", "generator"))]
    for k, i in enumerate(rng.sample(range(len(recs)), 12)):
        comp = k % 4
        if comp == 3:
            if rows[i]:
                rows[i][-1] = [E.R, E.R + 5, (1 << 256) - 1][k % 3]
            continue
        bad = bad2 if comp == 1 else bad1
        e = bad[k % len(bad)]
        off = (0, g1b, 3 * g1b)[comp]
        recs[i][off : off + len(e)] = e
    return b"".join(bytes(r) for r in recs), rows


@pytest.mark.parametrize("compressed", [True, False])
@pytest.mark.parametrize("m", [0, 1, 5])
def test_serialized_statuses_match_oracle(ctx, mixed, m, compressed):
    vkp, pts, inputs, kinds, _ = mixed[m]
    pvk = R.prepare_verifying_key(vkp, ctx)
    opvk = G.prepare_verifying_key(vkp)
    data, rows = _serialized_batch(pts, inputs, compressed, seed=m)
    rec = 192 if compressed else 384
    want = [G.status_serialized(opvk, data[i * rec : (i + 1) * rec], _xbytes([rows[i]]), compressed) for i in range(len(pts))]
    got = R.verify_proofs_serialized(pvk, _xbytes(rows), data, compressed)
    assert got.tolist() == want
    expect = {S.OK, G.REJECTED} | ({G.INPUT_NONCANONICAL} if m else set())
    assert expect <= set(want) and len(set(want) - expect) >= 2
    st, nv = ctx.groth16_verify_serialized(pvk.buf, m, _xbytes(rows), data, len(pts), compressed)
    assert nv == want.count(S.OK)


def test_serialized_refuses_bad_lengths(ctx, mixed):
    vkp, pts, inputs, kinds, _ = mixed[1]
    pvk = R.prepare_verifying_key(vkp, ctx)
    data, xb, n = _record(pts[0], True) + _record(pts[1], True), _xbytes(inputs[:2]), 2
    for d, x, cnt in ((data[:-1], xb, n), (data + b"\x00", xb, n), (data, xb[:-1], n), (data, xb + b"\x00" * 32, n),
                      (data, xb, n + 1), (data, xb, 1)):
        with pytest.raises(_lib.RippError) as e:
            ctx.groth16_verify_serialized(pvk.buf, 1, x, d, cnt, True)
        assert e.value.status == _lib.RIPP_ERR_ARG, (len(d), len(x), cnt)
    with pytest.raises(_lib.RippError) as e:  # the uncompressed mode reads 384-byte records
        ctx.groth16_verify_serialized(pvk.buf, 1, xb, data, n, False)
    assert e.value.status == _lib.RIPP_ERR_ARG


def test_keys_reused_and_two_keys_in_one_context(ctx, mixed):
    k1, k5 = R.prepare_verifying_key(mixed[1][0], ctx), R.prepare_verifying_key(mixed[5][0], ctx)
    for _ in range(2):
        for m, pvk in ((5, k5), (1, k1)):
            vkp, pts, inputs, kinds, want = mixed[m]
            assert R.verify_proofs(pvk, inputs, pts) == want, m
            st = R.verify_proofs_serialized(pvk, _xbytes(inputs), b"".join(_record(p, True) for p in pts), True)
            assert st.tolist() == [S.OK if w else G.REJECTED for w in want], m


# ---- large batches against the exponent-space truth ---------------------------------------------------------------
def _large(ctx, n, m, nfalse, seed):
    """n trapdoor-simulated proofs with nfalse tampered at seeded positions; points generated on the GPU."""
    sc, proofs, inputs = OS.groth16_instance_scalars(n, m, seed)
    vk, ic = sc["vk"], sc["ic"]
    proofs, inputs = list(proofs), [list(x) for x in inputs]
    rng = random.Random(seed)
    pos = rng.sample(range(n), nfalse)
    k = 0
    while k < len(pos):
        kind = G.GROTH16_TAMPER[k % 4]
        if kind == "b_swapped" and k + 1 < len(pos):
            G.groth16_tamper(vk, ic, proofs, inputs, kind, pos[k], pos[k + 1])
            k += 2
            continue
        G.groth16_tamper(vk, ic, proofs, inputs, "c_plus_g" if kind == "b_swapped" else kind, pos[k])
        k += 1
    truth = [G.groth16_exponent_verdict(vk, ic, p, x) for p, x in zip(proofs, inputs)]
    g1 = synth._gen_dev(ctx, 1, [vk["alpha"]] + ic).download((m + 2, 24))
    g2 = synth._gen_dev(ctx, 2, [vk["beta"], vk["gamma"], vk["delta"]]).download((3, 48))
    vk_words = np.concatenate([g1[0], g2[0], g2[1], g2[2]] + [g1[1 + j] for j in range(m + 1)])
    a = synth._gen_dev(ctx, 1, [p[0] for p in proofs])
    b = synth._gen_dev(ctx, 2, [p[1] for p in proofs])
    c = synth._gen_dev(ctx, 1, [p[2] for p in proofs])
    x = ctx.to_device(C.fr_vec_enc([v for row in inputs for v in row]))
    return vk_words, a, b, c, x, inputs, truth, sorted(pos)


def _verify_dev(ctx, vk_words, m, x, a, b, c, n):
    pvk = ctx.alloc(ctx.groth16_pvk_bytes(m))
    ctx.groth16_prepare_vk_dev(vk_words, m, pvk)
    out = ctx.alloc(n)
    ctx.groth16_verify_batch_dev(pvk, m, x, a, b, c, n, out)
    ctx.sync()
    return pvk, out.download(n, dtype=np.uint8)


def test_2p12_with_41_false_proofs(ctx):
    n, m = 1 << 12, 5
    vk_words, a, b, c, x, inputs, truth, pos = _large(ctx, n, m, 41, seed=12)
    assert truth.count(False) == 41 and [i for i, t in enumerate(truth) if not t] == pos
    pvk, got = _verify_dev(ctx, vk_words, m, x, a, b, c, n)
    assert got.tolist() == [int(t) for t in truth]
    data = SC.proof_records(a.download((n, 24)), b.download((n, 48)), c.download((n, 24)), True)
    st, nv = ctx.groth16_verify_serialized(pvk, m, _xbytes(inputs), data, n, True)
    assert st.tolist() == [S.OK if t else G.REJECTED for t in truth] and nv == n - 41


def test_2p16(ctx):
    n, m = 1 << 16, 5
    vk_words, a, b, c, x, inputs, truth, pos = _large(ctx, n, m, 41, seed=16)
    _, got = _verify_dev(ctx, vk_words, m, x, a, b, c, n)
    assert got.tolist() == [int(t) for t in truth]


# ---- tie-in with the aggregation ----------------------------------------------------------------------------------
def test_verdicts_and_aggregation(ctx):
    n, m = 1 << 6, 5
    inst = synth.tipp_instance_dev(ctx, n)
    _, got = _verify_dev(ctx, inst["vk"], m, ctx.to_device(inst["inputs"]), inst["a"], inst["b"], inst["c"], n)
    assert got.tolist() == [1] * n
    proof = ctx.tipp_aggregate_dev(inst["srs_g1"], inst["srs_g2"], inst["a"], inst["b"], inst["c"], n)
    assert ctx.tipp_verify_aggregate(inst["vsrs"], inst["vk"], inst["inputs"], proof)
    # one false proof: C + G at index 17
    vk, ic, proofs, inputs = synth.groth16_scalars(n)
    cs = [p[2] for p in proofs]
    cs[17] = (cs[17] + 1) % E.R
    c_bad = synth._gen_dev(ctx, 1, cs)
    _, got = _verify_dev(ctx, inst["vk"], m, ctx.to_device(inst["inputs"]), inst["a"], inst["b"], c_bad, n)
    assert [i for i, v in enumerate(got.tolist()) if v != 1] == [17]
    proof = ctx.tipp_aggregate_dev(inst["srs_g1"], inst["srs_g2"], inst["a"], inst["b"], c_bad, n)
    assert not ctx.tipp_verify_aggregate(inst["vsrs"], inst["vk"], inst["inputs"], proof)


# ---- ark-groth16's own verdicts, when tools/ark_golden has been run ------------------------------------------------
def test_golden_verdicts(ctx, mixed):
    """tools/ark_golden records ark-groth16's verify_proof on the m = 1 mixed batch (tests/golden/groth16_cases.txt) as
    groth16_verdict_<i>; the GPU verdicts equal them."""
    if not os.path.exists(GOLDEN):
        pytest.skip("tests/golden/ark_golden.json absent: run tools/ark_golden with a Rust toolchain (parity unpinned)")
    golden = json.load(open(GOLDEN))
    vkp, pts, inputs, kinds, _ = mixed[1]
    if "groth16_verdict_0" not in golden:
        pytest.skip("tests/golden/ark_golden.json predates the Groth16 verdicts: rerun tools/ark_golden with groth16_cases.txt")
    want = [golden["groth16_verdict_%d" % i] == "01" for i in range(len(pts))]
    assert R.verify_proofs(R.prepare_verifying_key(vkp, ctx), inputs, pts) == want
