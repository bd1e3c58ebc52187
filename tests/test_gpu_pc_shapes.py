"""The polynomial-commitment entry points (ripp_pc_commit_dev, ripp_pc_open_dev, ripp_pc_verify; csrc/poly_commit.cuh)
over the range of shapes they accept, trusted and transparent.

Small shapes (n rows of m) go byte for byte against the oracle (oracle/poly_commit.py) while n <= 16, and against a
composition of the older entry points above that, at every length class (empty, one coefficient, a row short, one row,
one short of full, full) and at the points 0, 1 and r - 1.  Large shapes cover each class of the row combination's
grouping (pc_scan.cuh row_groups: one group of several rows, many groups of several rows, and 2^16 rows of one, where
the group count is capped to fit the grid) against the composition: the pairing product, single MSMs, the resident
TIPA / GIPA provers on host-computed scalars, with the y_coms checked by a random linear combination."""
import functools
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
ALPHA, BETA = OS.scalar("pcs-alpha", 0), OS.scalar("pcs-beta", 0)
TRUSTED, TRANSPARENT = _lib.PC_TRUSTED, _lib.PC_TRANSPARENT
CK1, CK2 = "pcs-ck1", "pcs-ck2"
ORACLE_MAX_ROWS = 16  # the Python oracle's pairings grow with n


@pytest.fixture(scope="module")
def keys(ctx):
    """(kind, n, m, host_points) -> the device keys, made once per module."""
    cache = {}

    def get(kind, n, m, host_points=False):
        at = (kind, n, m, host_points)
        if at not in cache:
            if kind == TRUSTED:
                srs = PC.BivariatePolynomialCommitment.setup(n - 1, m - 1, ALPHA, BETA, ctx)
                cache[at] = {"B": PC.BivariatePolynomialCommitment, "key": srs, "vk": srs["v_srs"], "first": srs["kzg"][0],
                             "second": srs["ck"][0], "g2": srs["h_beta_powers"][0]}
            else:
                if host_points:  # the oracle's keys, uploaded
                    ck = PC.TransparentBivariatePolynomialCommitment.setup_from_points(OS.g1_points(CK1, m), OS.g2_points(CK2, n), ctx)
                else:
                    ck = {"first": (synth.g1_points_dev(ctx, CK1, m), m), "second": (synth.g2_points_dev(ctx, CK2, n), n)}
                cache[at] = {"B": PC.TransparentBivariatePolynomialCommitment, "key": ck, "vk": ck, "first": ck["first"][0],
                             "second": ck["second"][0], "g2": None}
        return cache[at]

    yield get
    cache.clear()


def _powers(s, n):
    out, cur = [], 1
    for _ in range(n):
        out.append(cur)
        cur = cur * s % R
    return out


def _msm(ctx, bases, words):
    """One ripp_msm_g1_dev over Montgomery scalar words (k, 8) -> affine words (24,)."""
    sc = ctx.to_device(np.ascontiguousarray(words, dtype=np.uint32))
    out = ctx.alloc(96)
    ctx.msm_g1_dev(bases, sc, len(words), out)
    ctx.sync()
    return out.download(24)


def _rejects(fn):
    try:
        return not fn()
    except _lib.RippError as e:
        return e.status == _lib.RIPP_ERR_ARG


def _random_words(seed, count):
    """count Montgomery Fr words, uniform below 2^224 * (r's top word): canonical, and no host encoding."""
    w = np.random.default_rng(seed).integers(0, 1 << 32, size=(count, 8), dtype=np.uint32)
    w[:, 7] %= np.uint32(R >> 224)
    return w


def _row_combinations(words, n, m, length, points):
    """[sum_i s^i row_i for s in points] of the coefficients `words` (length Montgomery Fr, row-major, row length m,
    zeros past length): Horner over the rows on the Montgomery integers, one division by 2^256 at the end."""
    raw = np.ascontiguousarray(words, dtype=np.uint32).tobytes()
    accs = [[0] * m for _ in points]
    for i in reversed(range(n)):
        lo, hi = i * m, min((i + 1) * m, length)
        row = [int.from_bytes(raw[32 * k:32 * k + 32], "little") for k in range(lo, hi)]
        row += [0] * (m - len(row))
        accs = [[(a * s + c) % R for a, c in zip(acc, row)] for acc, s in zip(accs, points)]
    return [[a * codec.RR_INV % R for a in acc] for acc in accs]


def _check_composition(ctx, kind, k, n, m, words, length, point, rho, y_eval, rlc, com, y_dev, proof, ev):
    """com, y_coms, proof and evaluation from the open against the older entry points on host-computed scalars.
    y_eval = sum_i x^i row_i and rlc = sum_i rho^i row_i come from the host."""
    x, y = point
    first, second = k["first"], k["second"]
    # the commitment: the n-pair product over the y_coms
    gt = ctx.alloc(576)
    ctx.pairing_ip_dev(y_dev, second, n, gt)
    ctx.sync()
    assert codec.gt_enc(com).tolist() == gt.download(144).tolist()
    # the y_coms: sum_i rho^i y_com_i == MSM(first tier, sum_i rho^i row_i), and single MSMs at sampled rows
    y_coms = y_dev.download((n, 24))
    assert np.array_equal(_msm(ctx, y_dev, codec.fr_vec_enc(_powers(rho, n))), _msm(ctx, first, codec.fr_vec_enc(rlc)))
    rnd = random.Random(rho)
    rows = {0, n - 1, min(max(length - 1, 0) // m, n - 1)}  # first, last, and the row where len ends
    while len(rows) < min(8, n):
        rows.add(rnd.randrange(n))
    for i in sorted(rows):
        sc = np.zeros((m, 8), dtype=np.uint32)
        lo, hi = i * m, min((i + 1) * m, length)
        if hi > lo:
            sc[:hi - lo] = words[lo:hi]
        assert np.array_equal(_msm(ctx, first, sc), y_coms[i]), i
    # the opening
    b = ctx.to_device(codec.fr_vec_enc(_powers(x, n)))
    ye_comm = codec.ser_g1(codec.g1_dec(_msm(ctx, first, codec.fr_vec_enc(y_eval))))
    if kind == TRUSTED:
        ip = ctx.tipa_prove_dev(_lib.GIPA_MULTIEXP_SSM, None, k["g2"], y_dev, b, second, None, n)
        q = OPC.quotient_by_linear(y_eval, y)
        want = ip + ye_comm + codec.ser_g1(codec.g1_dec(_msm(ctx, first, codec.fr_vec_enc(q + [0] * (m - len(q))))))
    else:
        ip2 = ctx.gipa_prove_dev(_lib.GIPA_MULTIEXP_SSM, y_dev, b, second, None, n)[0]
        a1, b1 = ctx.to_device(codec.fr_vec_enc(y_eval)), ctx.to_device(codec.fr_vec_enc(_powers(y, m)))
        ip1 = ctx.gipa_prove_dev(_lib.GIPA_SCALAR_SSM_G1, a1, b1, first, None, m)[0]
        want = ip2 + ye_comm + ip1
    assert proof == want
    assert ev == OPC.poly_eval(y_eval, y)


def _check_verify(ctx, kind, k, n, com, point, ev, proof, ev_swapped):
    """verify accepts the opening and rejects a wrong evaluation, the swapped point (unless f(y, x) = f(x, y): then the
    claim is true) and a one-bit flip of the proof (accept = 0 or undecodable bytes)."""
    def verify(pt, e, pf):
        return k["B"].verify(k["vk"], com, pt, e, pf, ctx)

    x, y = point
    assert verify(point, ev, proof)
    assert not verify(point, (ev + 1) % R, proof)
    if ev_swapped != ev:
        assert not verify((y, x), ev, proof)
    sites = [8] if n > 1 else []  # the first round's GT commitment (second tier)
    if kind == TRANSPARENT:
        # the first-tier GIPA's r_base = (a_base, b_base): a_base, the folded y_eval, carries the evaluation; b_base is
        # the structured message's, which the verifier recomputes from y and does not read (as the reference)
        sites.append(len(proof) - 64)
    for at in sites:
        bad = bytearray(proof)
        bad[at] ^= 0x01
        assert _rejects(lambda: verify(point, ev, bytes(bad))), at


# ---- small shapes ---------------------------------------------------------------------------------------------------
SMALL = [(2, 1), (2, 2), (4, 1), (2, 64), (64, 2), (16, 16), (1, 8), (1, 1)]


def _small_params():
    for n, m in SMALL:
        for kind in (TRUSTED, TRANSPARENT):
            if n == 1 and kind == TRUSTED:
                continue  # a one-row TIPA: test_trusted_one_row_is_rejected_before_any_launch
            yield pytest.param(kind, n, m, id="%s-%dx%d" % ("trusted" if kind == TRUSTED else "transparent", n, m))


@pytest.mark.parametrize("kind,n,m", list(_small_params()))
def test_small_shapes(ctx, keys, kind, n, m):
    B = PC.BivariatePolynomialCommitment if kind == TRUSTED else PC.TransparentBivariatePolynomialCommitment
    by_oracle = n <= ORACLE_MAX_ROWS
    k = keys(kind, n, m, host_points=by_oracle)
    if by_oracle:
        if kind == TRUSTED:
            OB, o_key, ser = OPC.BivariatePolynomialCommitment, OPC.BivariatePolynomialCommitment.setup(n - 1, m - 1, ALPHA, BETA), OPC.ser_opening_proof
        else:
            OB, o_key, ser = (OPC.TransparentBivariatePolynomialCommitment, (OS.g1_points(CK1, m), OS.g2_points(CK2, n)),
                              OPC.ser_transparent_opening_proof)
    rnd = random.Random(1000 * n + 10 * m + kind)
    vals = [rnd.randrange(R) for _ in range(n * m)]
    words = codec.fr_vec_enc(vals)
    lengths = sorted({0, 1, m - 1, m, n * m - 1, n * m})
    points = [(0, 0), (R - 1, 1), (1, rnd.randrange(R)), (rnd.randrange(R), 0), (rnd.randrange(R), R - 1),
              (rnd.randrange(R), rnd.randrange(R))]
    shift = SMALL.index((n, m))
    commits = {}
    for case in range(max(len(lengths), len(points))):
        length, point = lengths[case % len(lengths)], points[(case + shift) % len(points)]
        why = (length, point)
        rows = [(vals[:length] + [0] * (n * m - length))[i * m:(i + 1) * m] for i in range(n)]
        c = ctx.to_device(words[:length]) if length else None
        com, y_dev = B.commit_dev(k["key"], c, length, ctx)
        proof, ev = B.open_dev(k["key"], c, length, y_dev, point, ctx)
        assert ev == OPC.bivariate_evaluate(rows, point), why
        if by_oracle:
            if length not in commits:
                commits[length] = OB.commit(o_key, rows)
            o_com, o_y_coms = commits[length]
            assert com == o_com, why
            assert codec.g1_vec_dec(y_dev.download((n, 24))) == o_y_coms, why
            assert proof == ser(OB.open(o_key, rows, o_y_coms, point)), why
        else:
            rho = rnd.randrange(R)
            y_eval, rlc = _row_combinations(words, n, m, length, point[:1] + (rho,))
            _check_composition(ctx, kind, k, n, m, words, length, point, rho, y_eval, rlc, com, y_dev, proof, ev)
        _check_verify(ctx, kind, k, n, com, point, ev, proof, OPC.bivariate_evaluate(rows, point[::-1]))


def test_trusted_one_row_is_rejected_before_any_launch(ctx, keys):
    """A TIPA of one element has no challenge for its KZG opening (the reference panics at tipa/mod.rs:199): the
    trusted open of one row fails on its arguments, before the row combination or an MSM is launched.  Commit works."""
    one, two = codec.fr_enc(1), codec.fr_enc(2)
    for m in (1, 8):
        k = keys(TRANSPARENT, 1, m)  # any first-tier G1 and one G2 key
        c = ctx.to_device(codec.fr_vec_enc(list(range(1, m + 1))))
        y = ctx.alloc(96)
        ctx.pc_commit_dev(k["first"], m, k["second"], 1, c, m, y)
        ctx.sync()
        before = ctx.launches
        with pytest.raises(_lib.RippError) as e:
            ctx.pc_open_dev(TRUSTED, k["first"], m, k["second"], 1, k["second"], c, m, y, one, two)
        assert e.value.status == _lib.RIPP_ERR_ARG
        assert ctx.launches == before, m


# ---- large shapes: one per class of the row grouping ------------------------------------------------------------------
BIG = [
    # (n, m, len): row_groups gives
    ((1 << 16), 1, (1 << 16) - 1),        # G = 32768, R = 2: 2^16 groups would exceed the grid's 65535
    ((1 << 16), 4, (1 << 18) - 2),        # G = 16384, R = 4
    ((1 << 10), (1 << 8), 1 << 18),       # G = 256, R = 4
    (2, (1 << 16), (1 << 16) + 12345),    # G = 1, R = 2: k_pc_rows writes y_eval itself
    ((1 << 8), (1 << 16), (1 << 24) - 5),  # G = 1, R = 256, n m = 2^24 (the limit), a padded copy in commit
]


def _big_params():
    for n, m, length in BIG:
        marks = [pytest.mark.slow] if n * m == 1 << 24 else []
        for kind in (TRUSTED, TRANSPARENT):
            yield pytest.param(kind, n, m, length, marks=marks,
                               id="%s-%dx%d" % ("trusted" if kind == TRUSTED else "transparent", n, m))


@functools.lru_cache(maxsize=1)
def _big_case(n, m, length):
    """Coefficients, point and host row combinations of one large shape, shared by both kinds."""
    rnd = random.Random(n * 31 + m)
    words = _random_words(n * 31 + m, length)
    point, rho = (rnd.randrange(R), rnd.randrange(R)), rnd.randrange(R)
    y_eval, rlc = _row_combinations(words, n, m, length, (point[0], rho))
    return words, point, rho, y_eval, rlc


@pytest.mark.parametrize("kind,n,m,length", list(_big_params()))
def test_large_shape_equals_composition(ctx, keys, kind, n, m, length):
    words, point, rho, y_eval, rlc = _big_case(n, m, length)
    k = keys(kind, n, m)
    B = k["B"]
    c = ctx.to_device(words)
    com, y_dev = B.commit_dev(k["key"], c, length, ctx)
    proof, ev = B.open_dev(k["key"], c, length, y_dev, point, ctx)
    del c
    _check_composition(ctx, kind, k, n, m, words, length, point, rho, y_eval, rlc, com, y_dev, proof, ev)
    # random x != y: f(y, x) = f(x, y) with probability about 1 / r, so the swapped point is a false claim
    _check_verify(ctx, kind, k, n, com, point, ev, proof, None)
