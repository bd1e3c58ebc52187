"""Validated decoding of ark-serialize points on the GPU (csrc/deserialize.cu) and aggregate_proofs from the proofs'
bytes: status bytes and points equal the oracle's (oracle/serde.py de_g1 / de_g2, and its compiled restatement at
2^16 records), the aggregate equals the one from the same points passed as Montgomery limbs, invalid records are named."""
import numpy as np
import pytest

from oracle import serde as S
from oracle import protocols as O
from oracle import serde_cases as SC
from oracle import synth as OS
from oracle.cpu import binding as B
from oracle.cpu import serde_binding as SB
from ripp_b200 import _lib, codec as C, synth
from ripp_b200.ip_proofs import aggregate_proofs_serialized

pytestmark = pytest.mark.gpu

ENC = {1: C.g1_enc, 2: C.g2_enc}
DE = {1: S.de_g1, 2: S.de_g2}


def _dev_decode(ctx, group, data, n, stride, compressed, offset=0):
    buf = ctx.to_device(np.frombuffer(bytes(data), dtype=np.uint8).copy())
    words = 24 if group == 1 else 48
    out, st = ctx.alloc(n * 4 * words), ctx.alloc(max(n, 4))
    (ctx.g1_deserialize_dev if group == 1 else ctx.g2_deserialize_dev)(buf.ptr + offset, n, stride, compressed, out, st)
    ctx.sync()
    return out.download((n, words)), st.download(n, dtype=np.uint8)


@pytest.mark.parametrize("group", [1, 2])
@pytest.mark.parametrize("compressed", [True, False])
def test_status_and_points_match_oracle(ctx, group, compressed):
    batch = SC.mixed_batch(group, compressed, 160)
    pts, st = _dev_decode(ctx, group, b"".join(batch), len(batch), len(batch[0]), compressed)
    for i, b in enumerate(batch):
        want_pt, want_st = DE[group](b, compressed)
        assert st[i] == want_st, (i, S.STATUS_NAMES[st[i]], S.STATUS_NAMES[want_st])
        assert np.array_equal(pts[i], ENC[group](want_pt)), i
    assert set(st.tolist()) == set(range(5))


@pytest.mark.parametrize("compressed", [True, False])
def test_proof_record_stride(ctx, compressed):
    """A, B and C decoded in place from packed Proof records (stride = record size)."""
    n = 64
    a = SC.mixed_batch(1, compressed, n, seed=11)
    b = SC.mixed_batch(2, compressed, n, seed=12)
    c = SC.mixed_batch(1, compressed, n, seed=13)[::-1]
    g1b = len(a[0])
    rec = 4 * g1b
    data = b"".join(x + y + z for x, y, z in zip(a, b, c))
    for group, off, items in ((1, 0, a), (2, g1b, b), (1, 3 * g1b, c)):
        pts, st = _dev_decode(ctx, group, data, n, rec, compressed, offset=off)
        for i, e in enumerate(items):
            want_pt, want_st = DE[group](e, compressed)
            assert st[i] == want_st and np.array_equal(pts[i], ENC[group](want_pt)), (group, i)


def test_off_subgroup_points_rejected(ctx):
    for group, gen, ser in ((1, OS.g1_point_off_subgroup, (S.ser_g1_compressed, S.ser_g1)),
                            (2, OS.g2_point_off_subgroup, (S.ser_g2_compressed, S.ser_g2))):
        pts = [gen(seed) for seed in range(4)]
        for compressed, s in zip((True, False), ser):
            data = [s(p) for p in pts]
            out, st = _dev_decode(ctx, group, b"".join(data), len(data), len(data[0]), compressed)
            assert st.tolist() == [S.NOT_IN_SUBGROUP] * len(pts)
            assert not out.any()


def _srs(n):
    return O.tipa_setup(n, OS.scalar("srs-alpha", 0), OS.scalar("srs-beta", 0))


@pytest.mark.parametrize("n,compressed", [(16, True), (16, False), (64, True)])
def test_aggregate_serialized_bytes(ctx, n, compressed):
    srs = _srs(n)
    vk, proofs, inputs = OS.groth16_instance(n)
    data = SC.proof_records_from_points(proofs, compressed)
    got = aggregate_proofs_serialized((srs.g_alpha_powers, srs.h_beta_powers), data, compressed, ctx)
    a = ctx.to_device(C.g1_vec_enc([p[0] for p in proofs]))
    b = ctx.to_device(C.g2_vec_enc([p[1] for p in proofs]))
    c = ctx.to_device(C.g1_vec_enc([p[2] for p in proofs]))
    s1, s2 = ctx.to_device(C.g1_vec_enc(srs.g_alpha_powers)), ctx.to_device(C.g2_vec_enc(srs.h_beta_powers))
    assert got == ctx.tipp_aggregate_dev(s1, s2, a, b, c, n)
    if n == 16:  # the pure-Python oracle's own aggregate and verifier
        want = O.aggregate_proofs(srs, proofs)
        assert got == O.ser_aggregate_proof(want)
        assert O.verify_aggregate_proof(srs.get_verifier_key(), vk, inputs, want)
    else:
        be = B.CppBackend()
        srs_c = O.tipa_setup(n, OS.scalar("srs-alpha", 0), OS.scalar("srs-beta", 0), be=be)
        want = O.aggregate_proofs(srs_c, proofs, be=be)
        assert got == O.ser_aggregate_proof(want)
        assert O.verify_aggregate_proof(srs_c.get_verifier_key(), vk, inputs, want, be=be)


BAD = [  # (case name of serde_cases.named_cases, component, proof index, status text)
    ("flag_wrong_mode", "A", 3, "has invalid flag bits"),
    ("x_eq_p", "B", 5, "has a non-canonical coordinate (>= p)"),
    ("x_no_sqrt", "C", 0, "not on the curve"),
    ("off_subgroup", "B", 15, "not in the prime-order subgroup"),
    ("off_subgroup", "C", 9, "not in the prime-order subgroup"),
]


@pytest.mark.parametrize("case,comp,idx,text", BAD)
def test_invalid_record_is_named(ctx, case, comp, idx, text):
    n = 16
    srs = _srs(n)
    _, proofs, _ = OS.groth16_instance(n)
    recs = [bytearray(SC.proof_records_from_points([p], True)) for p in proofs]
    group = 2 if comp == "B" else 1
    bad = dict(SC.named_cases(group, True))[case]
    off = {"A": 0, "B": 48, "C": 144}[comp]
    recs[idx][off : off + len(bad)] = bad
    data = b"".join(bytes(r) for r in recs)
    with pytest.raises(_lib.RippError) as e:
        aggregate_proofs_serialized((srs.g_alpha_powers, srs.h_beta_powers), data, True, ctx)
    assert e.value.status == _lib.RIPP_ERR_ARG
    assert "proof %d: %s %s" % (idx, comp, text) in str(e.value), str(e.value)
    # the context is still usable: the same records without the bad element aggregate
    good = SC.proof_records_from_points(proofs, True)
    assert aggregate_proofs_serialized((srs.g_alpha_powers, srs.h_beta_powers), good, True, ctx)


def test_refuses_bad_lengths(ctx):
    n = 4
    srs = _srs(n)
    _, proofs, _ = OS.groth16_instance(n)
    s1, s2 = ctx.to_device(C.g1_vec_enc(srs.g_alpha_powers)), ctx.to_device(C.g2_vec_enc(srs.h_beta_powers))
    data = SC.proof_records_from_points(proofs, True)
    for blob, cnt, compressed, status in ((data[:-1], n, True, _lib.RIPP_ERR_ARG), (data + b"\x00", n, True, _lib.RIPP_ERR_ARG),
                                          (data, n + 1, True, _lib.RIPP_ERR_ARG), (data[: 3 * 192], 3, True, _lib.RIPP_ERR_NOT_POW2),
                                          (data[:192], 1, True, _lib.RIPP_ERR_ARG), (data, n, False, _lib.RIPP_ERR_ARG)):
        with pytest.raises(_lib.RippError) as e:
            ctx.tipp_aggregate_serialized(s1, s2, blob, cnt, compressed)
        assert e.value.status == status, (len(blob), cnt, str(e.value))


def test_aggregate_serialized_2p12_matches_tipp_aggregate(ctx):
    """configs[3] inputs (synth.tipp_instance_dev, 2^12 proofs) as compressed records: same AggregateProof bytes as
    ripp_tipp_aggregate on the Montgomery limbs, and the GPU verifier accepts them."""
    n = 1 << 12
    inst = synth.tipp_instance_dev(ctx, n)
    a_h, b_h, c_h = inst["a"].download((n, 24)), inst["b"].download((n, 48)), inst["c"].download((n, 24))
    data = SC.proof_records(a_h, b_h, c_h, True)
    got = ctx.tipp_aggregate_serialized(inst["srs_g1"], inst["srs_g2"], data, n, True)
    assert got == ctx.tipp_aggregate(inst["srs_g1"], inst["srs_g2"], a_h, b_h, c_h)
    assert ctx.tipp_verify_aggregate(inst["vsrs"], inst["vk"], inst["inputs"], got)


def test_status_2p16_records_match_cpu_restatement(ctx):
    """2^16 compressed Proof records with invalid elements injected at known indices: the GPU's status bytes and points
    equal oracle/cpu/serde_cpu.cpp's, component by component."""
    n = 1 << 16
    a_h = synth.g1_points_dev(ctx, "serde-a", n).download((n, 24))
    b_h = synth.g2_points_dev(ctx, "serde-b", n).download((n, 48))
    c_h = synth.g1_points_dev(ctx, "serde-c", n).download((n, 24))
    recs = bytearray(SC.proof_records(a_h, b_h, c_h, True))
    bad1 = [b for name, b in SC.named_cases(1, True) if not name.startswith(("valid", "identity", "generator"))]
    bad2 = [b for name, b in SC.named_cases(2, True) if not name.startswith(("valid", "identity", "generator"))]
    injected = {}
    for k, idx in enumerate(range(17, n, 4099)):
        comp = k % 3
        bad = bad2 if comp == 1 else bad1
        e = bad[k % len(bad)]
        off = 192 * idx + (0, 48, 144)[comp]
        recs[off : off + len(e)] = e
        injected[(idx, comp)] = e
    data = bytes(recs)
    for comp, group, off in ((0, 1, 0), (1, 2, 48), (2, 1, 144)):
        pts, st = _dev_decode(ctx, group, data, n, 192, True, offset=off)
        want_pts, want_st = SB.deserialize(group, data[off:], n, 192, True)
        assert np.array_equal(st, want_st), comp
        assert np.array_equal(pts, want_pts), comp
        bad_idx = {i for (i, c) in injected if c == comp}
        assert {int(i) for i in np.nonzero(st)[0]} == bad_idx
        src = (a_h, b_h, c_h)[comp]
        ok = np.array(sorted(set(range(n)) - bad_idx))
        assert np.array_equal(pts[ok], src[ok])
