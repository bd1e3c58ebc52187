"""Batched polynomial commitments (ripp_pc_commit_batch_dev, ripp_pc_open_batch_dev; csrc/pc_batch.cuh): every result of
a batch is byte for byte what the single entry points return for that polynomial alone, the proofs verify, the order of
a batch does not matter, the number of launches does not grow with the batch, and every argument error is raised before
anything is launched."""
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
ALPHA, BETA = OS.scalar("pcb-alpha", 0), OS.scalar("pcb-beta", 0)
TRUSTED, TRANSPARENT = _lib.PC_TRUSTED, _lib.PC_TRANSPARENT
CK1, CK2 = "pcb-ck1", "pcb-ck2"


@pytest.fixture(scope="module")
def keys(ctx):
    cache = {}

    def get(kind, n, m, host_points=False):
        at = (kind, n, m, host_points)
        if at not in cache:
            if kind == TRUSTED:
                srs = PC.BivariatePolynomialCommitment.setup(n - 1, m - 1, ALPHA, BETA, ctx)
                cache[at] = {"key": srs, "vk": srs["v_srs"], "first": srs["kzg"][0], "second": srs["ck"][0],
                             "g2": srs["h_beta_powers"][0]}
            else:
                if host_points:
                    ck = PC.TransparentBivariatePolynomialCommitment.setup_from_points(OS.g1_points(CK1, m), OS.g2_points(CK2, n), ctx)
                else:
                    ck = {"first": (synth.g1_points_dev(ctx, CK1, m), m), "second": (synth.g2_points_dev(ctx, CK2, n), n)}
                cache[at] = {"key": ck, "vk": ck, "first": ck["first"][0], "second": ck["second"][0], "g2": None}
        return cache[at]

    yield get
    cache.clear()


def _words(seed, count):
    """count canonical Montgomery Fr words without host encoding."""
    w = np.random.default_rng(seed).integers(0, 1 << 32, size=(max(count, 1), 8), dtype=np.uint32)
    w[:, 7] %= np.uint32(R >> 224)
    return w[:count]


def _instances(ctx, n, m, count, seed):
    """count polynomials of mixed lengths (0, 1, a row short, ending mid-row, full) at mixed points (0, 1, r - 1,
    random)."""
    rnd = random.Random(seed)
    nm = n * m
    classes = [0, 1, max(nm - m, 0), min(nm, m + m // 2 + 1) if n > 1 else max(nm // 2, 1), nm]
    lens = [min(classes[k % len(classes)], nm) for k in range(count)]
    pts = [0, 1, R - 1]
    xs = [pts[k % 3] if k < 3 else rnd.randrange(R) for k in range(count)]
    ys = [pts[(k + 1) % 3] if k < 4 else rnd.randrange(R) for k in range(count)]
    bufs = []
    for k in range(count):
        bufs.append(ctx.to_device(_words(seed * 1000 + k, lens[k])) if lens[k] else None)
    return bufs, lens, xs, ys


def _fr(vals):
    return np.stack([codec.fr_enc(v % R) for v in vals]) if vals else np.zeros((0, 8), np.uint32)


def _single(ctx, kind, k, n, m, buf, length, x, y):
    y_dev = ctx.alloc(n * 96)
    com = ctx.pc_commit_dev(k["first"], m, k["second"], n, buf, length, y_dev)
    proof, ev = ctx.pc_open_dev(kind, k["first"], m, k["second"], n, k["g2"], buf, length, y_dev, codec.fr_enc(x), codec.fr_enc(y))
    return com, y_dev.download((n, 24)), proof, ev


def _batch(ctx, kind, k, n, m, bufs, lens, xs, ys):
    count = len(bufs)
    y_dev = ctx.alloc(max(count, 1) * n * 96)
    coms = ctx.pc_commit_batch_dev(k["first"], m, k["second"], n, bufs, lens, y_dev)
    proofs, evs = ctx.pc_open_batch_dev(kind, k["first"], m, k["second"], n, k["g2"], bufs, lens, y_dev, _fr(xs), _fr(ys))
    return coms, y_dev.download((max(count, 1) * n, 24))[: count * n], proofs, evs


SHAPES = [(TRUSTED, 2, 8), (TRUSTED, 8, 8), (TRUSTED, 4, 1), (TRUSTED, 16, 4096),
          (TRANSPARENT, 2, 8), (TRANSPARENT, 8, 8), (TRANSPARENT, 4, 1), (TRANSPARENT, 16, 4096), (TRANSPARENT, 1, 8)]


@pytest.mark.parametrize("count", [1, 3, 8])
@pytest.mark.parametrize("kind,n,m", SHAPES)
def test_batch_equals_single_calls(ctx, keys, kind, n, m, count):
    k = keys(kind, n, m)
    bufs, lens, xs, ys = _instances(ctx, n, m, count, 7 * n + m + count)
    coms, y_coms, proofs, evs = _batch(ctx, kind, k, n, m, bufs, lens, xs, ys)
    assert len(proofs) == count and len(set(len(p) for p in proofs)) == 1
    for i in range(count):
        com, yc, proof, ev = _single(ctx, kind, k, n, m, bufs[i], lens[i], xs[i], ys[i])
        assert coms[i].tolist() == com.tolist(), i
        assert y_coms[i * n:(i + 1) * n].tolist() == yc.tolist(), i
        assert proofs[i] == proof, i
        assert evs[i].tolist() == ev.tolist(), i


@pytest.mark.parametrize("kind", [TRUSTED, TRANSPARENT])
def test_batch_against_oracle(ctx, keys, kind):
    n, m = (4, 4) if kind == TRUSTED else (2, 8)
    k = keys(kind, n, m, host_points=True)
    rnd = random.Random(kind)
    polys = [[[rnd.randrange(R) for _ in range(m)] for _ in range(n)], [[rnd.randrange(R) for _ in range(m - 1)]]]
    points = [(rnd.randrange(R), rnd.randrange(R)), (0, R - 1)]
    if kind == TRUSTED:
        B, OB, o_key, ser = PC.BivariatePolynomialCommitment, OPC.BivariatePolynomialCommitment, \
            OPC.BivariatePolynomialCommitment.setup(n - 1, m - 1, ALPHA, BETA), OPC.ser_opening_proof
    else:
        B, OB, o_key, ser = (PC.TransparentBivariatePolynomialCommitment, OPC.TransparentBivariatePolynomialCommitment,
                             (OS.g1_points(CK1, m), OS.g2_points(CK2, n)), OPC.ser_transparent_opening_proof)
    got = B.commit_batch(k["key"], polys, ctx)
    proofs = B.open_batch(k["key"], polys, [yc for _, yc in got], points, ctx)
    for p, (com, y_coms), point, proof in zip(polys, got, points, proofs):
        rows = [list(r) + [0] * (m - len(r)) for r in p] + [[0] * m] * (n - len(p))
        o_com, o_y_coms = OB.commit(o_key, rows)
        assert com == o_com and y_coms == o_y_coms
        assert proof == ser(OB.open(o_key, rows, o_y_coms, point))


def _verify(ctx, kind, k, n, m, com, x, y, ev, proof):
    vs = PC.vsrs_enc(k["vk"]) if kind == TRUSTED else None
    return ctx.pc_verify(kind, vs, k["first"], m, k["second"], n, com, codec.fr_enc(x), codec.fr_enc(y), ev, proof)


@pytest.mark.parametrize("kind,n,m", [(TRUSTED, 4, 8), (TRANSPARENT, 4, 8), (TRANSPARENT, 1, 4)])
def test_batched_proofs_verify(ctx, keys, kind, n, m):
    k = keys(kind, n, m)
    bufs, lens, xs, ys = _instances(ctx, n, m, 5, 99 + n)
    coms, _, proofs, evs = _batch(ctx, kind, k, n, m, bufs, lens, xs, ys)
    for i in range(5):
        assert _verify(ctx, kind, k, n, m, coms[i], xs[i], ys[i], evs[i], proofs[i]), i
        wrong = codec.fr_enc((codec.fr_dec(evs[i]) + 1) % R)
        assert not _verify(ctx, kind, k, n, m, coms[i], xs[i], ys[i], wrong, proofs[i]), i


@pytest.mark.parametrize("kind", [TRUSTED, TRANSPARENT])
def test_order_and_repeats(ctx, keys, kind):
    n, m = 4, 16
    k = keys(kind, n, m)
    bufs, lens, xs, ys = _instances(ctx, n, m, 5, 31 + kind)
    # the same pointer twice, one polynomial at two points
    bufs2, lens2 = bufs + [bufs[4], bufs[4]], lens + [lens[4], lens[4]]
    xs2, ys2 = xs + [xs[4], 12345], ys + [ys[4], 678]
    coms, y_coms, proofs, evs = _batch(ctx, kind, k, n, m, bufs2, lens2, xs2, ys2)
    assert coms[5].tolist() == coms[4].tolist() and proofs[5] == proofs[4] and evs[5].tolist() == evs[4].tolist()
    assert coms[6].tolist() == coms[4].tolist() and y_coms[6 * n:].tolist() == y_coms[4 * n:5 * n].tolist()
    single = _single(ctx, kind, k, n, m, bufs[4], lens[4], 12345, 678)
    assert proofs[6] == single[2] and evs[6].tolist() == single[3].tolist()
    # a permuted batch gives permuted outputs
    perm = [3, 0, 4, 1, 2]
    pc, py, pp, pe = _batch(ctx, kind, k, n, m, [bufs[p] for p in perm], [lens[p] for p in perm], [xs[p] for p in perm],
                            [ys[p] for p in perm])
    for i, p in enumerate(perm):
        assert pc[i].tolist() == coms[p].tolist() and pp[i] == proofs[p] and pe[i].tolist() == evs[p].tolist()
        assert py[i * n:(i + 1) * n].tolist() == y_coms[p * n:(p + 1) * n].tolist()


@pytest.mark.parametrize("kind,n,m", [(TRUSTED, 8, 64), (TRANSPARENT, 8, 64), (TRANSPARENT, 1, 64)])
def test_launch_count_does_not_grow_with_count(ctx, keys, kind, n, m):
    k = keys(kind, n, m)
    counts = {}
    for count in (2, 16):
        bufs, lens, xs, ys = _instances(ctx, n, m, count, 5 + count)
        y_dev = ctx.alloc(count * n * 96)
        a = ctx.launches
        ctx.pc_commit_batch_dev(k["first"], m, k["second"], n, bufs, lens, y_dev)
        b = ctx.launches
        ctx.pc_open_batch_dev(kind, k["first"], m, k["second"], n, k["g2"], bufs, lens, y_dev, _fr(xs), _fr(ys))
        counts[count] = (b - a, ctx.launches - b)
    assert counts[16][0] <= counts[2][0] and counts[16][1] <= counts[2][1], counts


def test_transparent_at_the_coefficient_limit(ctx, keys):
    """n = 1, m = 256, count = 2^16: count n m = 2^24, against single calls on a seeded sample."""
    n, m, count = 1, 256, 1 << 16
    k = keys(TRANSPARENT, n, m)
    big = ctx.to_device(_words(4242, 4096 * m))
    rnd = random.Random(4242)
    lens = [rnd.choice([0, 1, m // 2 + 3, m]) for _ in range(count)]
    bufs = [big.ptr + (i % 4096) * m * 32 if lens[i] else None for i in range(count)]
    xs = [rnd.randrange(R) for _ in range(count)]
    ys = [rnd.randrange(R) for _ in range(count)]
    coms, y_coms, proofs, evs = _batch(ctx, TRANSPARENT, k, n, m, bufs, lens, xs, ys)
    for i in sorted(set(rnd.randrange(count) for _ in range(6)) | {0, count - 1}):
        com, yc, proof, ev = _single(ctx, TRANSPARENT, k, n, m, bufs[i], lens[i], xs[i], ys[i])
        assert coms[i].tolist() == com.tolist() and y_coms[i].tolist() == yc[0].tolist(), i
        assert proofs[i] == proof and evs[i].tolist() == ev.tolist(), i


def test_trusted_univariate_degree_65535(ctx):
    """16 univariate polynomials of degree 65535 (n = 16 rows of 4096), against single calls."""
    U = PC.UnivariatePolynomialCommitment
    srs = U.setup(65535, ALPHA, BETA, ctx)
    n, m = srs["ck"][1], srs["kzg"][1]
    bufs = [ctx.to_device(_words(77 + i, n * m)) for i in range(16)]
    lens = [n * m] * 15 + [n * m - 5]
    rnd = random.Random(77)
    zs = [rnd.randrange(R) for _ in range(16)]
    coms, y_dev = U.commit_batch_dev(srs, bufs, lens, ctx)
    proofs, evs = U.open_batch_dev(srs, bufs, lens, y_dev, zs, ctx)
    for i in range(16):
        com, y1 = U.commit_dev(srs, bufs[i], lens[i], ctx)
        proof, ev = U.open_dev(srs, bufs[i], lens[i], y1, zs[i], ctx)
        assert coms[i] == com and proofs[i] == proof and evs[i] == ev, i
    assert U.verify(srs["v_srs"], 65535, coms[0], zs[0], evs[0], proofs[0], ctx)


def test_argument_errors_launch_nothing(ctx, keys):
    n, m = 4, 8
    kt, kp = keys(TRUSTED, n, m), keys(TRANSPARENT, n, m)
    bufs, lens, xs, ys = _instances(ctx, n, m, 2, 3)
    y_dev = ctx.alloc(2 * n * 96)
    X, Y = _fr(xs), _fr(ys)

    def commit(first=kp["first"], mm=m, second=kp["second"], nn=n, b=bufs, ln=lens):
        return ctx.pc_commit_batch_dev(first, mm, second, nn, b, ln, y_dev)

    def open_(kind=TRANSPARENT, k=kp, mm=m, nn=n, b=bufs, ln=lens, g2=None):
        return ctx.pc_open_batch_dev(kind, k["first"], mm, k["second"], nn, g2 if g2 is not None else k["g2"], b, ln, y_dev, X, Y)

    cases = [
        (_lib.RIPP_ERR_ARG, lambda: commit(first=None)),
        (_lib.RIPP_ERR_ARG, lambda: commit(b=[None, bufs[1]], ln=[5, lens[1]])),
        (_lib.RIPP_ERR_NOT_POW2, lambda: commit(mm=6)),
        (_lib.RIPP_ERR_NOT_POW2, lambda: commit(nn=3)),
        (_lib.RIPP_ERR_ARG, lambda: commit(ln=[lens[0], n * m + 1])),
        (_lib.RIPP_ERR_ARG, lambda: commit(nn=1 << 16, b=bufs, ln=[0, 0], mm=1)),
        (_lib.RIPP_ERR_ARG, lambda: commit(nn=1 << 12, mm=1 << 12, ln=[0, 0])),
        (_lib.RIPP_ERR_ARG, lambda: open_(kind=7)),
        (_lib.RIPP_ERR_ARG, lambda: ctx.pc_open_batch_dev(TRUSTED, kt["first"], m, kt["second"], n, None, bufs, lens, y_dev, X, Y)),
        (_lib.RIPP_ERR_NOT_POW2, lambda: open_(mm=12)),
        (_lib.RIPP_ERR_ARG, lambda: open_(kind=TRUSTED, k=kt, nn=1)),
        (_lib.RIPP_ERR_ARG, lambda: open_(ln=[n * m + 1, 0])),
        (_lib.RIPP_ERR_ARG, lambda: open_(nn=1 << 16, mm=1, ln=[0, 0])),
    ]
    for status, fn in cases:
        before = ctx.launches
        with pytest.raises(_lib.RippError) as e:
            fn()
        assert e.value.status == status, (status, e.value)
        assert ctx.launches == before
    # a too small output buffer: ARG with the length set; count 0: OK with length 0
    import ctypes
    cnt, ptrs, lv = ctx._pc_batch_args(bufs, lens)
    plen = ctypes.c_size_t()
    before = ctx.launches
    st = _lib.lib().ripp_pc_open_batch_dev(ctx.handle, TRANSPARENT, _lib._p(kp["first"]), ctypes.c_size_t(m), _lib._p(kp["second"]),
                                           ctypes.c_size_t(n), None, ctypes.c_size_t(2), ptrs, _lib._p(lv), _lib._p(y_dev),
                                           _lib._p(X), _lib._p(Y), _lib._p(np.zeros(16, np.uint8)), ctypes.c_size_t(16),
                                           ctypes.byref(plen), None)
    assert st == _lib.RIPP_ERR_ARG and plen.value > 0 and ctx.launches == before
    plen.value = 99
    st = _lib.lib().ripp_pc_open_batch_dev(ctx.handle, TRANSPARENT, _lib._p(kp["first"]), ctypes.c_size_t(m), _lib._p(kp["second"]),
                                           ctypes.c_size_t(n), None, ctypes.c_size_t(0), None, None, None, None, None, None,
                                           ctypes.c_size_t(0), ctypes.byref(plen), None)
    assert st == _lib.RIPP_OK and plen.value == 0 and ctx.launches == before
    assert len(ctx.pc_commit_batch_dev(kp["first"], m, kp["second"], n, [], [], None)) == 0
    assert ctx.launches == before
