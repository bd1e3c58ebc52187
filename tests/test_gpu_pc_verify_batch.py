"""Batched verification of polynomial-commitment openings (ripp_pc_verify_batch; csrc/pc_verify_batch.cuh): every
status is what ripp_pc_verify reports for that opening alone, for valid, false, malformed and off-subgroup openings of
both kinds; no status depends on the rest of the batch; the launch count does not grow with the batch; every argument
error is returned in the documented order before anything is launched; and full-size openings decide as the single
verifier does."""
import ctypes
import random

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import synth as OS
from oracle.encoding import ser_g1, ser_g2
from ripp_b200 import _lib, codec, synth
from ripp_b200 import poly_commit as PC
from ripp_b200.ip_proofs import AGG_MALFORMED, AGG_NOT_IN_SUBGROUP, AGG_OK, AGG_REJECTED, vsrs_enc

pytestmark = pytest.mark.gpu
R = E.R
ALPHA, BETA = OS.scalar("pcv-alpha", 0), OS.scalar("pcv-beta", 0)
TRUSTED, TRANSPARENT = _lib.PC_TRUSTED, _lib.PC_TRANSPARENT
CK1, CK2 = "pcv-ck1", "pcv-ck2"
SHAPE = {TRUSTED: (4, 8), TRANSPARENT: (4, 16)}
OTHER = {TRUSTED: (2, 32), TRANSPARENT: (4, 8)}  # trusted: another SRS, same VerifierSRS; transparent: another first tier


@pytest.fixture(scope="module")
def keys(ctx):
    cache = {}

    def get(kind, n, m):
        if (kind, n, m) not in cache:
            if kind == TRUSTED:
                srs = PC.BivariatePolynomialCommitment.setup(n - 1, m - 1, ALPHA, BETA, ctx)
                cache[kind, n, m] = {"key": srs, "vsrs": vsrs_enc(srs["v_srs"]), "first": srs["kzg"][0], "second": srs["ck"][0],
                                     "g2": srs["h_beta_powers"][0], "n": n, "m": m}
            else:
                ck = {"first": (synth.g1_points_dev(ctx, CK1, m), m), "second": (synth.g2_points_dev(ctx, CK2, n), n)}
                cache[kind, n, m] = {"key": ck, "vsrs": None, "first": ck["first"][0], "second": ck["second"][0], "g2": None,
                                     "n": n, "m": m}
        return cache[kind, n, m]

    yield get
    cache.clear()


def _words(seed, count):
    w = np.random.default_rng(seed).integers(0, 1 << 32, size=(max(count, 1), 8), dtype=np.uint32)
    w[:, 7] %= np.uint32(R >> 224)
    return w[:count]


def _open(ctx, kind, k, lens, points, seed):
    """commit_batch + open_batch of polynomials of the given lengths.  -> list of (com, x, y, eval, proof)"""
    n, m = k["n"], k["m"]
    bufs = [ctx.to_device(_words(seed * 100 + i, ln)) if ln else None for i, ln in enumerate(lens)]
    y_dev = ctx.alloc(len(lens) * n * 96)
    coms = ctx.pc_commit_batch_dev(k["first"], m, k["second"], n, bufs, lens, y_dev)
    xs = np.stack([codec.fr_enc(x % R) for x, _ in points])
    ys = np.stack([codec.fr_enc(y % R) for _, y in points])
    proofs, evs = ctx.pc_open_batch_dev(kind, k["first"], m, k["second"], n, k["g2"], bufs, lens, y_dev, xs, ys)
    return [[coms[i], xs[i], ys[i], evs[i], proofs[i]] for i in range(len(lens))]


def _fr_plus_one(w):
    return codec.fr_enc((codec.fr_dec(w) + 1) % R)


def _splice(proof, at, data):
    return proof[:at] + data + proof[at + len(data):]


def _second_len(n):
    return 8 + (n.bit_length() - 1) * 2 * (576 + 32 + 8 + 96) + 96 + 32


def _members(ctx, keys, kind):
    """The mixed batch of one kind: (name, [com, x, y, eval, proof]) pairs."""
    n, m = SHAPE[kind]
    k = keys(kind, n, m)
    rnd = random.Random(kind + 17)
    pts = [(rnd.randrange(R), rnd.randrange(R)), (0, R - 1), (1, rnd.randrange(R))]
    good = _open(ctx, kind, k, [n * m, m + 3, n * m - 1], pts, 5 + kind)
    z = rnd.randrange(R)
    uni = _open(ctx, kind, k, [n * m - 2], [(pow(z, m, R), z)], 9 + kind)[0]  # a univariate opening: (z^m, z)
    on, om = OTHER[kind]
    other = _open(ctx, kind, keys(kind, on, om), [on * om], [(rnd.randrange(R), rnd.randrange(R))], 13 + kind)[0]
    out = [("valid %d" % i, g) for i, g in enumerate(good)] + [("univariate", uni)]
    com, x, y, ev, proof = good[0]
    out.append(("wrong eval", [com, x, y, _fr_plus_one(ev), proof]))
    out.append(("other point", [com, good[1][1], good[1][2], ev, proof]))
    out.append(("other commitment", [good[1][0], x, y, ev, proof]))
    flip = bytearray(proof)
    flip[8 + 5] ^= 1  # the first round's first GT element
    out.append(("flipped GT byte", [com, x, y, ev, bytes(flip)]))
    out.append(("truncated", [com, x, y, ev, proof[:-1]]))
    out.append(("empty", [com, x, y, ev, b""]))
    off1 = ser_g1(OS.g1_point_off_subgroup())
    ye_at = len(proof) - 192 if kind == TRUSTED else _second_len(n)
    out.append(("off-subgroup y_eval_comm", [com, x, y, ev, _splice(proof, ye_at, off1)]))
    out.append(("off-subgroup com_gt", [codec.gt_enc(OS.gt_cyclotomic_off_subgroup()), x, y, ev, proof]))
    if kind == TRUSTED:
        # the final key's KZG proof is the TIPA proof's last element, before y_eval_comm || kzg_proof
        out.append(("off-subgroup final-key proof", [com, x, y, ev, _splice(proof, len(proof) - 192 - 192, ser_g2(OS.g2_point_off_subgroup()))]))
        out.append(("another SRS shape", other))
        kz = bytearray(proof)
        kz[-1] ^= 1  # kzg_proof's y coordinate: off the curve
        out.append(("kzg proof off the curve", [com, x, y, ev, bytes(kz)]))
    else:
        out.append(("wrong round count", other))
        # the zero polynomial (a0 = O) with r_base's b0 changed: the single verifier still accepts
        zc, zx, zy, zev, zp = _open(ctx, kind, k, [0], [(rnd.randrange(R), rnd.randrange(R))], 21)[0]
        b0_at = _second_len(n) - 32
        b0 = int.from_bytes(zp[b0_at:b0_at + 32], "little")
        out.append(("a0 = O, b0 changed", [zc, zx, zy, zev, _splice(zp, b0_at, ((b0 + 1) % R).to_bytes(32, "little"))]))
    return k, out


def _single(ctx, kind, k, member):
    com, x, y, ev, proof = member
    try:
        ok = ctx.pc_verify(kind, k["vsrs"], k["first"], k["m"], k["second"], k["n"], com, x, y, ev, proof)
        return AGG_OK if ok else AGG_REJECTED
    except _lib.RippError as e:
        assert e.status == _lib.RIPP_ERR_ARG
        return AGG_NOT_IN_SUBGROUP if "subgroup" in str(e) else AGG_MALFORMED


def _raw(ctx, kind, k, members, n=None, m=None, proof_lens=None, proofs_len=None, **null):
    """ripp_pc_verify_batch through ctypes; a keyword argument `name=1` passes NULL for that pointer.  -> (return code,
    statuses, *n_accepted)"""
    count = len(members)
    coms = np.ascontiguousarray(np.stack([c[0] for c in members]) if count else np.zeros((1, 144), np.uint32))
    fr = [np.ascontiguousarray(np.stack([c[i] for c in members]) if count else np.zeros((1, 8), np.uint32)) for i in (1, 2, 3)]
    data = b"".join(c[4] for c in members)
    buf = np.frombuffer(data + b"\0", dtype=np.uint8).copy()
    ln = np.array(proof_lens if proof_lens is not None else [len(c[4]) for c in members] or [0], dtype=np.uintp)
    st = np.full(max(count, 1), 0xff, dtype=np.uint8)
    acc = ctypes.c_size_t(12345)
    args = {"vsrs": k["vsrs"], "first": k["first"], "second": k["second"], "coms": coms, "x": fr[0], "y": fr[1], "ev": fr[2],
            "proofs": buf, "lens": ln, "status": st}
    for name in null:
        args[name] = None
    p = {a: _lib._p(v) for a, v in args.items()}
    rc = _lib.lib().ripp_pc_verify_batch(
        None if null.get("ctx_null") else ctx.handle, int(kind), p["vsrs"], p["first"], ctypes.c_size_t(k["m"] if m is None else m),
        p["second"], ctypes.c_size_t(k["n"] if n is None else n), ctypes.c_size_t(count), p["coms"], p["x"], p["y"], p["ev"],
        p["proofs"], ctypes.c_size_t(len(data) if proofs_len is None else proofs_len), p["lens"], p["status"],
        None if null.get("acc_null") else ctypes.byref(acc))
    return rc, st[:count].tolist(), acc.value


@pytest.mark.parametrize("kind", [TRUSTED, TRANSPARENT])
def test_mixed_batch_matches_single_verifier(ctx, keys, kind):
    k, members = _members(ctx, keys, kind)
    want = [_single(ctx, kind, k, mem) for _, mem in members]
    names = [nm for nm, _ in members]
    expect = {"valid 0": AGG_OK, "valid 1": AGG_OK, "valid 2": AGG_OK, "univariate": AGG_OK, "wrong eval": AGG_REJECTED,
              "other point": AGG_REJECTED, "other commitment": AGG_REJECTED, "truncated": AGG_MALFORMED, "empty": AGG_MALFORMED,
              "off-subgroup y_eval_comm": AGG_NOT_IN_SUBGROUP, "off-subgroup com_gt": AGG_NOT_IN_SUBGROUP,
              "off-subgroup final-key proof": AGG_NOT_IN_SUBGROUP, "another SRS shape": AGG_OK,
              "kzg proof off the curve": AGG_MALFORMED, "wrong round count": AGG_REJECTED, "a0 = O, b0 changed": AGG_OK}
    for nm, w in zip(names, want):
        if nm in expect:
            assert w == expect[nm], (nm, w)
    rc, st, acc = _raw(ctx, kind, k, [mem for _, mem in members])
    assert rc == _lib.RIPP_OK
    assert st == want, list(zip(names, st, want))
    assert acc == sum(s == AGG_OK for s in want)
    # the Python wrapper of the class returns the same statuses
    evs = [codec.fr_dec(mem[3]) for _, mem in members]
    pts = [(codec.fr_dec(mem[1]), codec.fr_dec(mem[2])) for _, mem in members]
    coms = [codec.gt_dec(mem[0]) for _, mem in members]
    proofs = [mem[4] for _, mem in members]
    if kind == TRUSTED:
        got = PC.BivariatePolynomialCommitment.verify_batch(k["key"]["v_srs"], coms, pts, evs, proofs, ctx)
    else:
        got = PC.TransparentBivariatePolynomialCommitment.verify_batch(k["key"], coms, pts, evs, proofs, ctx)
    assert got.dtype == np.uint8 and got.tolist() == want


@pytest.mark.parametrize("kind", [TRUSTED, TRANSPARENT])
def test_univariate_wrappers(ctx, keys, kind):
    """The univariate classes map z_k to (z_k^(y_degree + 1), z_k), as their verify does."""
    if kind == TRUSTED:
        U, degree = PC.UnivariatePolynomialCommitment, 63
        srs = U.setup(degree, ALPHA, BETA, ctx)
        key, vkey = srs, srs["v_srs"]
    else:
        U, degree = PC.TransparentUnivariatePolynomialCommitment, 63
        xd, yd = U.bivariate_degrees(degree)
        key = vkey = PC.TransparentBivariatePolynomialCommitment.setup_from_points(OS.g1_points(CK1, yd + 1), OS.g2_points(CK2, xd + 1), ctx)
    rnd = random.Random(kind + 40)
    polys = [[rnd.randrange(R) for _ in range(degree + 1)], [rnd.randrange(R) for _ in range(10)]]
    committed = U.commit_batch(key, polys, ctx)
    zs = [rnd.randrange(R), 0]
    proofs = U.open_batch(key, polys, [c[1] for c in committed], zs, ctx)
    evs = [sum(c * pow(z, i, R) for i, c in enumerate(p)) % R for p, z in zip(polys, zs)]
    coms = [c[0] for c in committed]
    args = (vkey, degree) if kind == TRUSTED else (vkey,)
    got = U.verify_batch(*args, coms + coms[:1], zs + [zs[1]], evs + [evs[0]], proofs + proofs[:1], ctx)
    want = [int(not U.verify(*args, c, z, e, p, ctx)) * AGG_REJECTED
            for c, z, e, p in zip(coms + coms[:1], zs + [zs[1]], evs + [evs[0]], proofs + proofs[:1])]
    assert got.tolist() == want == [AGG_OK, AGG_OK, AGG_REJECTED]


@pytest.mark.parametrize("kind", [TRUSTED, TRANSPARENT])
def test_statuses_do_not_depend_on_the_batch(ctx, keys, kind):
    k, members = _members(ctx, keys, kind)
    mems = [mem for _, mem in members]
    _, st, _ = _raw(ctx, kind, k, mems)
    perm = list(range(len(mems)))
    random.Random(3).shuffle(perm)
    _, st_p, _ = _raw(ctx, kind, k, [mems[i] for i in perm])
    assert st_p == [st[i] for i in perm]
    for i, mem in enumerate(mems):
        rc, one, acc = _raw(ctx, kind, k, [mem])
        assert rc == _lib.RIPP_OK and one == [st[i]] == [_single(ctx, kind, k, mem)], members[i][0]
        assert acc == int(st[i] == AGG_OK)


@pytest.mark.parametrize("kind", [TRUSTED, TRANSPARENT])
def test_launch_count_does_not_grow(ctx, keys, kind):
    n, m = SHAPE[kind]
    k = keys(kind, n, m)
    rnd = random.Random(kind + 50)
    good = _open(ctx, kind, k, [n * m] * 4, [(rnd.randrange(R), rnd.randrange(R)) for _ in range(4)], 30 + kind)
    big = [good[i % 4] for i in range(16)]
    big[5] = [big[5][0], big[5][1], big[5][2], _fr_plus_one(big[5][3]), big[5][4]]
    _raw(ctx, kind, k, big)  # sizes the scratch
    counts = []
    for mem in (big[:2], big):
        before = ctx.launches
        rc, st, _ = _raw(ctx, kind, k, mem)
        counts.append(ctx.launches - before)
        assert rc == _lib.RIPP_OK and st.count(AGG_OK) == len(mem) - (mem is big)
    assert counts[0] == counts[1] > 0


def test_argument_errors(ctx, keys):
    kt, kp = keys(TRUSTED, *SHAPE[TRUSTED]), keys(TRANSPARENT, *SHAPE[TRANSPARENT])
    _, members = _members(ctx, keys, TRUSTED)
    one = [members[0][1]]
    ARG, NP2, OK = _lib.RIPP_ERR_ARG, _lib.RIPP_ERR_NOT_POW2, _lib.RIPP_OK
    before = ctx.launches
    # 1. null ctx or n_accepted, or a bad kind (before count == 0)
    assert _raw(ctx, TRUSTED, kt, one, ctx_null=True)[0] == ARG
    assert _raw(ctx, TRUSTED, kt, one, acc_null=True)[0] == ARG
    assert _raw(ctx, 2, kt, [])[0] == ARG
    # 2. count == 0, other pointers null
    assert _raw(ctx, TRUSTED, kt, [], vsrs=1, coms=1, x=1, y=1, ev=1, proofs=1, lens=1, status=1) == (OK, [], 0)
    # 3. other null pointers (before the missing VerifierSRS)
    for name in ("coms", "x", "y", "ev", "proofs", "lens", "status"):
        assert _raw(ctx, TRUSTED, kt, one, vsrs=1, **{name: 1})[0] == ARG, name
    # 4. trusted without vsrs
    assert _raw(ctx, TRUSTED, kt, one, vsrs=1)[0] == ARG
    # 5. transparent: null keys, then the shape (NOT_POW2 before ARG)
    assert _raw(ctx, TRANSPARENT, kp, one, first=1, n=3)[0] == ARG
    assert _raw(ctx, TRANSPARENT, kp, one, second=1)[0] == ARG
    assert _raw(ctx, TRANSPARENT, kp, one, n=3, m=1 << 25)[0] == NP2
    assert _raw(ctx, TRANSPARENT, kp, one, n=1 << 17, m=1)[0] == ARG
    assert _raw(ctx, TRANSPARENT, kp, one, n=1 << 16, m=1 << 9)[0] == ARG
    # 6. the batch limits: count > 2^16; transparent count n or count m > 2^24 (empty proofs: the limits come first)
    empty = [one[0][:4] + [b""]]
    assert _raw(ctx, TRUSTED, kt, empty * ((1 << 16) + 1))[0] == ARG
    assert _raw(ctx, TRANSPARENT, kp, empty * 512, n=1 << 16, m=1)[0] == ARG
    assert _raw(ctx, TRANSPARENT, kp, empty * 32, n=1, m=1 << 20)[0] == ARG
    # 7. proof_lens that do not sum to proofs_len
    plen = len(one[0][4])
    assert _raw(ctx, TRUSTED, kt, one, proofs_len=plen - 1)[0] == ARG
    assert _raw(ctx, TRUSTED, kt, one, proofs_len=plen + 1)[0] == ARG
    assert _raw(ctx, TRUSTED, kt, one * 2, proof_lens=[plen, plen + 1], proofs_len=2 * plen)[0] == ARG
    assert ctx.launches == before
    # proof_lens that sum right but split the bytes elsewhere are data: two malformed openings
    assert _raw(ctx, TRUSTED, kt, one * 2, proof_lens=[plen + 1, plen - 1]) == (OK, [AGG_MALFORMED] * 2, 0)


@pytest.mark.parametrize("kind,n,m", [(TRUSTED, 64, 16384), (TRANSPARENT, 256, 4096)])
def test_full_size(ctx, keys, kind, n, m):
    """Four openings of 2^20 coefficients, two valid and two wrong: the single verifier's statuses."""
    k = keys(kind, n, m)
    rnd = random.Random(n + m)
    mems = _open(ctx, kind, k, [n * m, n * m - 5, n * m, n * m - 1000], [(rnd.randrange(R), rnd.randrange(R)) for _ in range(4)],
                 60 + kind)
    mems[2][3] = _fr_plus_one(mems[2][3])
    mems[3][1] = mems[0][1]
    want = [_single(ctx, kind, k, mem) for mem in mems]
    assert want == [AGG_OK, AGG_OK, AGG_REJECTED, AGG_REJECTED]
    rc, st, acc = _raw(ctx, kind, k, mems)
    assert rc == _lib.RIPP_OK and st == want and acc == 2
