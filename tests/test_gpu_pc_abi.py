"""The polynomial-commitment entry points of the C ABI (ripp_fr_div_linear_dev, ripp_pc_kzg_*, ripp_pc_commit_dev,
ripp_pc_open_dev, ripp_pc_verify; csrc/poly_commit.cuh) against the oracle at the reference's test sizes, and against a
composition of the older primitive entry points (one ripp_msm_g1_dev per Y polynomial, ripp_pairing_ip_dev, the
resident TIPA / GIPA provers on host-computed scalars) at univariate degree 65535."""
import random

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import poly_commit as OPC
from oracle import synth as OS
from ripp_b200 import _lib, codec, synth
from ripp_b200 import poly_commit as PC

pytestmark = pytest.mark.gpu
R = E.R
ALPHA, BETA = OS.scalar("pca-alpha", 0), OS.scalar("pca-beta", 0)


def _fr_dev(ctx, vals):
    return ctx.to_device(codec.fr_vec_enc(vals)) if vals else None


def _div(ctx, coeffs, z):
    c = _fr_dev(ctx, coeffs)
    q = ctx.alloc(max(len(coeffs) - 1, 1) * 32)
    ev = ctx.alloc(32)
    ctx.fr_div_linear_dev(c, len(coeffs), codec.fr_enc(z), q, ev)
    ctx.sync()
    nq = max(len(coeffs) - 1, 0)
    return (codec.fr_vec_dec(q.download((nq, 8))) if nq else []), codec.fr_dec(ev.download(8))


@pytest.mark.parametrize("n", [0, 1, 2, 31, 32, 33, 1023, 1024, 1025, 32769])
def test_div_linear_matches_oracle(ctx, n):
    rnd = random.Random(n)
    coeffs = [rnd.randrange(R) for _ in range(n)]
    for z in (0, 1, R - 1, rnd.randrange(R)):
        q, ev = _div(ctx, coeffs, z)
        assert q == OPC.quotient_by_linear(coeffs, z), (n, z)
        assert ev == OPC.poly_eval(coeffs, z), (n, z)


def test_div_linear_at_2_20_plus_3(ctx):
    n = (1 << 20) + 3
    rnd = random.Random(3)
    coeffs = [rnd.randrange(R) for _ in range(n)]
    z = rnd.randrange(R)
    q, ev = _div(ctx, coeffs, z)
    assert q == OPC.quotient_by_linear(coeffs, z)
    assert ev == OPC.poly_eval(coeffs, z)


def test_kzg_matches_oracle(ctx):
    powers, v_srs = PC.KZG.setup(9, ALPHA, BETA, ctx)
    o_powers, _ = OPC.KZG.setup(9, ALPHA, BETA)
    rnd = random.Random(1)
    vs = PC.vsrs_enc(v_srs)
    for n in (0, 1, 2, 8, 10):
        poly = [rnd.randrange(R) for _ in range(n)]
        z = rnd.randrange(R)
        com, proof = PC.KZG.commit(powers, poly, ctx), PC.KZG.open(powers, poly, z, ctx)
        assert com == OPC.KZG.commit(o_powers, poly) and proof == OPC.KZG.open(o_powers, poly, z), n
        if n == 0:
            assert com is None and proof is None  # the identity
        if n == 1:
            assert proof is None  # an empty quotient
        ev = OPC.poly_eval(poly, z)
        # the evaluation comes back from the open
        c = _fr_dev(ctx, poly)
        out, evd = ctx.alloc(96), ctx.alloc(32)
        ctx.pc_kzg_open_dev(powers[0], powers[1], c, n, codec.fr_enc(z), out, evd)
        assert codec.fr_dec(evd.download(8)) == ev
        assert ctx.pc_kzg_verify(vs, codec.g1_enc(com), codec.fr_enc(z), codec.fr_enc(ev), codec.g1_enc(proof))
        assert not ctx.pc_kzg_verify(vs, codec.g1_enc(com), codec.fr_enc(z), codec.fr_enc((ev + 1) % R), codec.g1_enc(proof))


def _trusted(ctx, xd=7, yd=7):
    return PC.BivariatePolynomialCommitment.setup(xd, yd, ALPHA, BETA, ctx), OPC.BivariatePolynomialCommitment.setup(xd, yd, ALPHA, BETA)


@pytest.mark.parametrize("rows,row_len", [(8, 8), (5, 8), (8, 3)])
def test_trusted_bivariate_matches_oracle(ctx, rows, row_len):
    B, OB = PC.BivariatePolynomialCommitment, OPC.BivariatePolynomialCommitment
    srs, o_srs = _trusted(ctx)
    rnd = random.Random(rows * 10 + row_len)
    ys = [[rnd.randrange(R) for _ in range(row_len)] for _ in range(rows)]
    com, y_coms = B.commit(srs, ys, ctx)
    o_com, o_y_coms = OB.commit(o_srs, ys)
    assert com == o_com and y_coms == o_y_coms
    point = (rnd.randrange(R), rnd.randrange(R))
    proof = B.open(srs, ys, y_coms, point, ctx)
    assert proof == OPC.ser_opening_proof(OB.open(o_srs, ys, o_y_coms, point))
    ev = OPC.bivariate_evaluate(ys, point)
    assert B.verify(srs["v_srs"], com, point, ev, proof, ctx)
    assert not B.verify(srs["v_srs"], com, point, (ev + 1) % R, proof, ctx)


def test_univariate_len_ending_mid_row(ctx):
    """A univariate polynomial of 29 coefficients in the 8 x 8 layout: rows 3 .. 7 partly or wholly zero."""
    srs, o_srs = _trusted(ctx)
    rnd = random.Random(29)
    poly = [rnd.randrange(R) for _ in range(29)]
    rows = PC.UnivariatePolynomialCommitment.bivariate_form((7, 7), poly)
    c = _fr_dev(ctx, poly)
    com, y_dev = PC.BivariatePolynomialCommitment.commit_dev(srs, c, len(poly), ctx)
    o_com, o_y_coms = OPC.BivariatePolynomialCommitment.commit(o_srs, rows)
    assert com == o_com and codec.g1_vec_dec(y_dev.download((8, 24))) == o_y_coms
    point = (rnd.randrange(R), rnd.randrange(R))
    proof, ev = PC.BivariatePolynomialCommitment.open_dev(srs, c, len(poly), y_dev, point, ctx)
    assert proof == OPC.ser_opening_proof(OPC.BivariatePolynomialCommitment.open(o_srs, rows, o_y_coms, point))
    assert ev == OPC.bivariate_evaluate(rows, point)
    # transparent, same layout
    first, second = OS.g1_points("pca-ck1", 8), OS.g2_points("pca-ck2", 8)
    ck = PC.TransparentBivariatePolynomialCommitment.setup_from_points(first, second, ctx)
    OT = OPC.TransparentBivariatePolynomialCommitment
    com, y_dev = PC.TransparentBivariatePolynomialCommitment.commit_dev(ck, c, len(poly), ctx)
    o_com, o_y_coms = OT.commit((first, second), rows)
    assert com == o_com and codec.g1_vec_dec(y_dev.download((8, 24))) == o_y_coms
    proof, ev = PC.TransparentBivariatePolynomialCommitment.open_dev(ck, c, len(poly), y_dev, point, ctx)
    assert proof == OPC.ser_transparent_opening_proof(OT.open((first, second), rows, o_y_coms, point))
    assert ev == OPC.bivariate_evaluate(rows, point)


@pytest.mark.parametrize("rows", [8, 6])
def test_transparent_bivariate_matches_oracle(ctx, rows):
    T, OT = PC.TransparentBivariatePolynomialCommitment, OPC.TransparentBivariatePolynomialCommitment
    first, second = OS.g1_points("pca-ck1", 8), OS.g2_points("pca-ck2", 8)
    ck = T.setup_from_points(first, second, ctx)
    rnd = random.Random(rows)
    ys = [[rnd.randrange(R) for _ in range(8)] for _ in range(rows)]
    com, y_coms = T.commit(ck, ys, ctx)
    o_com, o_y_coms = OT.commit((first, second), ys)
    assert com == o_com and y_coms == o_y_coms
    point = (rnd.randrange(R), rnd.randrange(R))
    proof = T.open(ck, ys, y_coms, point, ctx)
    assert proof == OPC.ser_transparent_opening_proof(OT.open((first, second), ys, o_y_coms, point))
    ev = OPC.bivariate_evaluate(ys, point)
    assert T.verify(ck, com, point, ev, proof, ctx)
    assert not T.verify(ck, com, point, (ev + 1) % R, proof, ctx)


# ---- the same proofs composed from the older primitive entry points ------------------------------------------------
def _powers(s, n):
    out, cur = [], 1
    for _ in range(n):
        out.append(cur)
        cur = cur * s % R
    return out


def _msm(ctx, bases, vals):
    sc = ctx.to_device(codec.fr_vec_enc(vals))
    out = ctx.alloc(96)
    ctx.msm_g1_dev(bases, sc, len(vals), out)
    ctx.sync()
    return out.download(24)


def _composed(ctx, kind, first, m, second, n, srs_g2, poly, point):
    """com, y_coms, proof bytes by per-row MSMs, one pairing product, host scalars and the resident provers."""
    x, y = point
    flat = poly + [0] * (n * m - len(poly))
    rows = [flat[i * m:(i + 1) * m] for i in range(n)]
    y_coms = np.stack([_msm(ctx, first, r) for r in rows])
    yd = ctx.to_device(y_coms)
    gt = ctx.alloc(576)
    ctx.pairing_ip_dev(yd, second, n, gt)
    ctx.sync()
    px = _powers(x, n)
    y_eval = [sum(px[i] * rows[i][j] for i in range(n)) % R for j in range(m)]
    ye_comm = codec.ser_g1(codec.g1_dec(_msm(ctx, first, y_eval)))
    b = ctx.to_device(codec.fr_vec_enc(px))
    if kind == _lib.PC_TRUSTED:
        ip = ctx.tipa_prove_dev(_lib.GIPA_MULTIEXP_SSM, None, srs_g2, yd, b, second, None, n)
        q = OPC.quotient_by_linear(y_eval, y)
        proof = ip + ye_comm + codec.ser_g1(codec.g1_dec(_msm(ctx, first, q + [0] * (m - len(q)))))
    else:
        ip2 = ctx.gipa_prove_dev(_lib.GIPA_MULTIEXP_SSM, yd, b, second, None, n)[0]
        a1, b1 = ctx.to_device(codec.fr_vec_enc(y_eval)), ctx.to_device(codec.fr_vec_enc(_powers(y, m)))
        ip1 = ctx.gipa_prove_dev(_lib.GIPA_SCALAR_SSM_G1, a1, b1, first, None, m)[0]
        proof = ip2 + ye_comm + ip1
    return gt.download(144), y_coms, proof


def _rejects(fn):
    try:
        return not fn()
    except _lib.RippError as e:
        return e.status == _lib.RIPP_ERR_ARG


@pytest.mark.parametrize("kind", [_lib.PC_TRUSTED, _lib.PC_TRANSPARENT])
def test_univariate_degree_65535_equals_composition(ctx, kind):
    degree = 65535
    rnd = random.Random(kind)
    if kind == _lib.PC_TRUSTED:
        U = PC.UnivariatePolynomialCommitment
        srs = U.setup(degree, ALPHA, BETA, ctx)
        xd, yd = U.degrees_from_srs(srs)
        first, second, srs_g2 = srs["kzg"][0], srs["ck"][0], srs["h_beta_powers"][0]
        key = srs
    else:
        U = PC.TransparentUnivariatePolynomialCommitment
        xd, yd = U.bivariate_degrees(degree)
        key = {"first": (synth.g1_points_dev(ctx, "pca-ck1", yd + 1), yd + 1),
               "second": (synth.g2_points_dev(ctx, "pca-ck2", xd + 1), xd + 1)}
        first, second, srs_g2 = key["first"][0], key["second"][0], None
    n, m = xd + 1, yd + 1
    assert n * m == degree + 1
    poly = [rnd.randrange(R) for _ in range(degree + 1)]
    z = rnd.randrange(R)
    c = _fr_dev(ctx, poly)
    com, y_dev = U.commit_dev(key, c, len(poly), ctx)
    proof, ev = U.open_dev(key, c, len(poly), y_dev, z, ctx)
    w_gt, w_coms, w_proof = _composed(ctx, kind, first, m, second, n, srs_g2, poly, (pow(z, m, R), z))
    assert codec.gt_enc(com).tolist() == w_gt.tolist()
    assert np.array_equal(y_dev.download((n, 24)), w_coms)
    assert proof == w_proof
    assert ev == OPC.poly_eval(poly, z)
    if kind == _lib.PC_TRUSTED:
        verify = lambda cm, pt, e, pf: U.verify(srs["v_srs"], degree, cm, pt, e, pf, ctx)  # noqa: E731
    else:
        verify = lambda cm, pt, e, pf: U.verify(key, cm, pt, e, pf, ctx)  # noqa: E731
    assert verify(com, z, ev, proof)
    assert not verify(com, z, (ev + 1) % R, proof)
    assert not verify(com, (z + 1) % R, ev, proof)
    # swapped coordinates of the bivariate point
    x = pow(z, m, R)
    B = PC.BivariatePolynomialCommitment if kind == _lib.PC_TRUSTED else PC.TransparentBivariatePolynomialCommitment
    vk = srs["v_srs"] if kind == _lib.PC_TRUSTED else key
    assert B.verify(vk, com, (x, z), ev, proof, ctx)
    assert not B.verify(vk, com, (z, x), ev, proof, ctx)
    for at in (9, len(proof) // 2, len(proof) - 40):
        bad = bytearray(proof)
        bad[at] ^= 0x01
        assert _rejects(lambda: verify(com, z, ev, bytes(bad))), at


def test_commit_launch_count_does_not_depend_on_rows(ctx):
    """The n Y polynomials are one segmented MSM: besides the n-pair product (whose reduction tree has log n depth, as
    every ripp_pairing_ip_dev of n pairs), commit launches the same kernels for 4 and for 64 rows."""
    m = 64
    first = synth.g1_points_dev(ctx, "pca-ck1", m)
    counts = []
    for n in (4, 64):
        second = synth.g2_points_dev(ctx, "pca-ck2", n)
        c = _fr_dev(ctx, [random.Random(n).randrange(R) for _ in range(n * m - 5)])
        y, gt = ctx.alloc(n * 96), ctx.alloc(576)
        ctx.pc_commit_dev(first, m, second, n, c, n * m - 5, y)  # warm-up: workspaces, child contexts
        before = ctx.launches
        ctx.pc_commit_dev(first, m, second, n, c, n * m - 5, y)
        mid = ctx.launches
        ctx.pairing_ip_dev(y, second, n, gt)
        ctx.sync()
        counts.append((mid - before) - (ctx.launches - mid))
    assert counts[0] == counts[1], counts


def _status(fn):
    with pytest.raises(_lib.RippError) as e:
        fn()
    return e.value.status


def test_argument_errors(ctx):
    m, n = 8, 8
    first, second = synth.g1_points_dev(ctx, "pca-ck1", m), synth.g2_points_dev(ctx, "pca-ck2", n)
    c = _fr_dev(ctx, list(range(1, n * m + 1)))
    y = ctx.alloc(1 << 20)
    one = codec.fr_enc(1)
    NP2, ARG = _lib.RIPP_ERR_NOT_POW2, _lib.RIPP_ERR_ARG
    assert _status(lambda: ctx.pc_commit_dev(first, m, second, 6, c, 8, y)) == NP2
    assert _status(lambda: ctx.pc_commit_dev(first, 6, second, n, c, 8, y)) == NP2
    assert _status(lambda: ctx.pc_commit_dev(first, m, second, 0, c, 0, y)) == NP2
    assert _status(lambda: ctx.pc_commit_dev(first, m, second, 1 << 17, c, 8, y)) == ARG
    assert _status(lambda: ctx.pc_commit_dev(first, 1 << 20, second, 32, c, 8, y)) == ARG
    assert _status(lambda: ctx.pc_commit_dev(first, m, second, n, c, n * m + 1, y)) == ARG
    assert _status(lambda: ctx.pc_commit_dev(None, m, second, n, c, 8, y)) == ARG
    assert _status(lambda: ctx.pc_commit_dev(first, m, second, n, None, 8, y)) == ARG
    assert _status(lambda: ctx.pc_commit_dev(first, m, second, n, c, 8, None)) == ARG
    for kind in (_lib.PC_TRUSTED, _lib.PC_TRANSPARENT):
        g2 = second if kind == _lib.PC_TRUSTED else None
        assert _status(lambda: ctx.pc_open_dev(kind, first, m, second, 6, g2, c, 8, y, one, one)) == NP2
        assert _status(lambda: ctx.pc_open_dev(kind, first, 12, second, n, g2, c, 8, y, one, one)) == NP2
        assert _status(lambda: ctx.pc_open_dev(kind, first, m, second, 1 << 17, g2, c, 8, y, one, one)) == ARG
        assert _status(lambda: ctx.pc_open_dev(kind, first, m, second, n, g2, c, n * m + 1, y, one, one)) == ARG
        assert _status(lambda: ctx.pc_open_dev(kind, first, m, second, n, g2, c, 8, None, one, one)) == ARG
        assert _status(lambda: ctx.pc_open_dev(kind, first, m, second, n, g2, c, 8, y, None, one)) == ARG
    assert _status(lambda: ctx.pc_open_dev(_lib.PC_TRUSTED, first, m, second, n, None, c, 8, y, one, one)) == ARG
    assert _status(lambda: ctx.pc_open_dev(7, first, m, second, n, second, c, 8, y, one, one)) == ARG
    # undecodable proof bytes
    gt = codec.gt_enc(E.multi_pairing([E.G1_GEN], [E.G2_GEN]))
    vs = PC.vsrs_enc({"g": E.G1_GEN, "h": E.G2_GEN, "g_beta": E.G1_GEN, "h_alpha": E.G2_GEN})
    for kind in (_lib.PC_TRUSTED, _lib.PC_TRANSPARENT):
        assert _status(lambda: ctx.pc_verify(kind, vs, first, m, second, n, gt, one, one, one, b"\x01" * 100)) == ARG
        assert _status(lambda: ctx.pc_verify(kind, vs, first, m, second, n, gt, one, one, one, b"\xff" * 5000)) == ARG
    assert _status(lambda: ctx.pc_verify(_lib.PC_TRANSPARENT, None, first, 6, second, n, gt, one, one, one, b"\0" * 5000)) == NP2
    # KZG and the division
    assert _status(lambda: ctx.pc_kzg_commit_dev(first, m, c, m + 1, y)) == ARG
    assert _status(lambda: ctx.pc_kzg_open_dev(first, m, c, m + 1, one, y)) == ARG
    assert _status(lambda: ctx.pc_kzg_open_dev(first, m, None, 4, one, y)) == ARG
    assert _status(lambda: ctx.fr_div_linear_dev(c, 4, one, None)) == ARG
    assert _status(lambda: ctx.fr_div_linear_dev(None, 4, one, y)) == ARG
    assert _status(lambda: ctx.fr_div_linear_dev(c, 4, None, y)) == ARG
