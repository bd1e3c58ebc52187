"""ripp_tipp_verify_aggregate_batch: many aggregates under one VerifierSRS and one VerifyingKey in one call.  Every
status must be what ripp_tipp_verify_aggregate reports for that aggregate alone, whatever else is in the batch."""
import random

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import synth as OS
from oracle.encoding import ser_g1, ser_g2, ser_gt
from ripp_b200 import _lib, codec as C
from ripp_b200.ip_proofs import (AGG_MALFORMED, AGG_NOT_IN_SUBGROUP, AGG_OK, AGG_REJECTED, aggregate_proofs, verify_aggregate_proofs,
                                 vk_enc, vsrs_enc)
from test_gpu_protocols import _srs

pytestmark = pytest.mark.gpu
NMAX = 32


@pytest.fixture(scope="module")
def inst(ctx):
    """One vk, one VerifierSRS (the SRS of every size shares g, h, g_beta, h_alpha) and aggregates of prefixes and
    permutations of the seeded instance's proofs."""
    vk, proofs, inputs = OS.groth16_instance(NMAX)
    vs = _srs(2).get_verifier_key()
    srs = {}

    def agg(idx):
        n = len(idx)
        if n not in srs:
            s = _srs(n)
            assert s.get_verifier_key() == vs
            srs[n] = (s.g_alpha_powers, s.h_beta_powers)
        rows = [list(inputs[i]) for i in idx]
        return rows, aggregate_proofs(srs[n], [proofs[i] for i in idx], ctx)

    return {"vk": vk, "vs": vs, "agg": agg, "vsrs": vsrs_enc(vs), "vkw": np.ascontiguousarray(vk_enc(vk))}


def _enc(rows):
    return np.ascontiguousarray(np.stack([C.fr_vec_enc(r) for r in rows]).reshape(len(rows), len(rows[0]), 8))


def _single(ctx, inst, rows, proof):
    """ripp_tipp_verify_aggregate's outcome as a ripp_agg_status."""
    try:
        return AGG_OK if ctx.tipp_verify_aggregate(inst["vsrs"], inst["vkw"], _enc(rows), proof) else AGG_REJECTED
    except _lib.RippError as e:
        assert e.status == _lib.RIPP_ERR_ARG
        return AGG_NOT_IN_SUBGROUP if "subgroup" in str(e) else AGG_MALFORMED


def _batch(ctx, inst, members):
    return ctx.tipp_verify_aggregate_batch(inst["vsrs"], inst["vkw"], [_enc(r) for r, _ in members], [p for _, p in members])


def _flip(b, i):
    b = bytearray(b)
    b[i] ^= 1
    return bytes(b)


def _splice(b, at, new):
    return b[:at] + new + b[at + len(new):]


@pytest.fixture(scope="module")
def mixed(inst):
    rnd = random.Random(5)
    agg = inst["agg"]
    members = [agg(list(range(n))) for n in (2, 4, 8, NMAX)]
    for n in (8, NMAX):
        perm = list(range(n))
        rnd.shuffle(perm)
        members.append(agg(perm))
    rows4, p4 = members[1]
    rows2, p2 = members[0]
    bad_rows = [list(r) for r in rows4]
    bad_rows[1][2] = (bad_rows[1][2] + 1) % E.R
    members.append((bad_rows, p4))  # wrong public input
    members.append((rows4, _flip(p4, 0)))  # com_a
    members.append((rows4, _flip(p4, 3 * 576)))  # ip_ab
    members.append((rows2, p2[:-1]))  # truncated
    off1, off2, offt = OS.g1_point_off_subgroup(), OS.g2_point_off_subgroup(), OS.gt_cyclotomic_off_subgroup()
    members.append((rows4, _splice(p4, 4 * 576, ser_g1(off1))))  # agg_c
    members.append((rows4, _splice(p4, len(p4) - 192, ser_g2(off2))))  # the C proof's final_ck_proof
    members.append((rows4, _splice(p4, 576, ser_gt(offt))))  # com_b
    perm_rows = [list(r) for r in members[5][0]]
    perm_rows[-1][0] = (perm_rows[-1][0] + 1) % E.R
    members.append((perm_rows, members[5][1]))  # permuted aggregate of 32, wrong input row
    return members


def test_mixed_batch_matches_single_verifier(ctx, inst, mixed):
    want = [_single(ctx, inst, r, p) for r, p in mixed]
    # a flipped GT byte leaves GT's subgroup (NOT_IN_SUBGROUP) unless it happens to land in it (REJECTED)
    assert want[7] in (AGG_NOT_IN_SUBGROUP, AGG_REJECTED) and want[8] in (AGG_NOT_IN_SUBGROUP, AGG_REJECTED)
    assert want[:7] + want[9:] == [AGG_OK] * 6 + [AGG_REJECTED, AGG_MALFORMED] + [AGG_NOT_IN_SUBGROUP] * 3 + [AGG_REJECTED]
    got = _batch(ctx, inst, mixed)
    assert got.dtype == np.uint8 and list(got) == want
    # n_accepted through the C entry point
    import ctypes

    ns = np.array([len(r) for r, _ in mixed], dtype=np.uintp)
    lens = np.array([len(p) for _, p in mixed], dtype=np.uintp)
    inp = np.ascontiguousarray(np.concatenate([_enc(r).reshape(-1) for r, _ in mixed]))
    data = b"".join(p for _, p in mixed)
    buf = np.frombuffer(data, dtype=np.uint8).copy()
    st = np.zeros(len(mixed), dtype=np.uint8)
    acc = ctypes.c_size_t()
    _lib.check(_lib.lib().ripp_tipp_verify_aggregate_batch(
        ctx.handle, _lib._p(inst["vsrs"]), _lib._p(inst["vkw"]), ctypes.c_size_t(5), ctypes.c_size_t(len(mixed)), _lib._p(ns),
        _lib._p(inp), _lib._p(buf), ctypes.c_size_t(len(data)), _lib._p(lens), _lib._p(st), ctypes.byref(acc)))
    assert list(st) == want and acc.value == want.count(AGG_OK)


def test_statuses_do_not_depend_on_the_batch(ctx, inst, mixed):
    want = list(_batch(ctx, inst, mixed))
    perm = list(range(len(mixed)))
    random.Random(9).shuffle(perm)
    got = _batch(ctx, inst, [mixed[i] for i in perm])
    assert list(got) == [want[i] for i in perm]
    for i in (0, 3, 6, 9, 10, 12):  # K = 1
        assert list(_batch(ctx, inst, [mixed[i]])) == [_single(ctx, inst, *mixed[i])]


def test_launch_count_does_not_grow_with_the_batch(ctx, inst, mixed):
    eights = [mixed[2], mixed[4]]
    counts = []
    for k in (2, 16):
        members = [eights[i % 2] for i in range(k)]
        _batch(ctx, inst, members)  # scratch sized for k
        before = ctx.launches
        assert list(_batch(ctx, inst, members)) == [AGG_OK] * k
        counts.append(ctx.launches - before)
    assert counts[0] == counts[1], counts


def test_python_api_and_errors(ctx, inst, mixed):
    vk, vs = inst["vk"], inst["vs"]
    proofs = [p for _, p in mixed]
    st = verify_aggregate_proofs(vs, vk, [r for r, _ in mixed], proofs, ctx)
    assert list(st) == list(_batch(ctx, inst, mixed))
    assert len(ctx.tipp_verify_aggregate_batch(inst["vsrs"], inst["vkw"], [], [])) == 0  # count == 0
    import ctypes

    def call(m=5, ns=(2,), lens=None, data=None, null_status=False):
        data = mixed[0][1] if data is None else data
        lens = np.array([len(data)] if lens is None else lens, dtype=np.uintp)
        ns = np.array(ns, dtype=np.uintp)
        inp = np.zeros(max(1, int(ns.sum())) * max(m, 1) * 8, dtype=np.uint32)
        buf = np.frombuffer(data, dtype=np.uint8).copy()
        st = np.zeros(len(ns), dtype=np.uint8)
        acc = ctypes.c_size_t()
        return _lib.lib().ripp_tipp_verify_aggregate_batch(
            ctx.handle, _lib._p(inst["vsrs"]), _lib._p(inst["vkw"]), ctypes.c_size_t(m), ctypes.c_size_t(len(ns)), _lib._p(ns),
            _lib._p(inp), _lib._p(buf), ctypes.c_size_t(len(data)), _lib._p(lens), None if null_status else _lib._p(st),
            ctypes.byref(acc))

    assert call() == _lib.RIPP_OK
    assert call(ns=(0,)) == _lib.RIPP_ERR_ARG
    assert call(m=0) == _lib.RIPP_ERR_ARG
    assert call(m=1025) == _lib.RIPP_ERR_ARG
    assert call(lens=[len(mixed[0][1]) - 1]) == _lib.RIPP_ERR_ARG
    assert call(lens=[len(mixed[0][1]) + 1]) == _lib.RIPP_ERR_ARG
    assert call(null_status=True) == _lib.RIPP_ERR_ARG


def test_full_size(ctx):
    """Four aggregates of 2^12 proofs: the seeded instance, a permutation of it, and each with one wrong input row."""
    from ripp_b200 import synth

    n = 1 << 12
    t = synth.tipp_instance_dev(ctx, n)
    a, b, c = t["a"].download((n, 24)), t["b"].download((n, 48)), t["c"].download((n, 24))
    perm = np.random.default_rng(3).permutation(n)
    pa, pb, pc = ctx.to_device(a[perm]), ctx.to_device(b[perm]), ctx.to_device(c[perm])
    proof = ctx.tipp_aggregate_dev(t["srs_g1"], t["srs_g2"], t["a"], t["b"], t["c"], n)
    proof_p = ctx.tipp_aggregate_dev(t["srs_g1"], t["srs_g2"], pa, pb, pc, n)
    rows, rows_p = t["inputs"], np.ascontiguousarray(t["inputs"][perm])
    bad = rows.copy()
    bad[7, 0] = C.fr_enc((C.fr_dec(bad[7, 0]) + 1) % E.R)
    bad_p = rows_p.copy()
    bad_p[n - 1, 0] = C.fr_enc((C.fr_dec(bad_p[n - 1, 0]) + 1) % E.R)
    members = [(rows, proof), (rows_p, proof_p), (bad, proof), (bad_p, proof_p)]
    want = [ctx.tipp_verify_aggregate(t["vsrs"], t["vk"], r, p) for r, p in members]
    assert want == [True, True, False, False]
    got = ctx.tipp_verify_aggregate_batch(t["vsrs"], t["vk"], [r for r, _ in members], [p for _, p in members])
    assert list(got) == [AGG_OK, AGG_OK, AGG_REJECTED, AGG_REJECTED]
