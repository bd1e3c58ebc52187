"""ripp_tipp_aggregate_batch_dev: many batches of Groth16 proofs under one SRS in one call, their GIPA rounds in lock
step.  Proof k must be byte for byte what ripp_tipp_aggregate_dev returns for batch k alone.  Also the segmented MSM
entry points (ripp_msm_g{1,2}_batch_dev) against one MSM per segment."""
import ctypes

import numpy as np
import pytest

from oracle import bls12_381 as E
from oracle import protocols as O
from oracle import synth as OS
from ripp_b200 import _lib, codec as C, synth
from ripp_b200.ip_proofs import AGG_OK, aggregate_proofs, aggregate_proofs_batch
from test_gpu_protocols import _srs

pytestmark = pytest.mark.gpu
NPOOL = 512


@pytest.fixture(scope="module")
def pool(ctx):
    """NPOOL simulated Groth16 proofs and an SRS of 2 NPOOL - 1 powers (long enough for every n here), on the GPU."""
    t = synth.tipp_instance_dev(ctx, NPOOL)
    t["ha"], t["hb"], t["hc"] = t["a"].download((NPOOL, 24)), t["b"].download((NPOOL, 48)), t["c"].download((NPOOL, 24))
    return t


def _pick(pool, idx):
    return pool["ha"][idx], pool["hb"][idx], pool["hc"][idx]


def _single(ctx, pool, idx):
    a, b, c = (ctx.to_device(x) for x in _pick(pool, idx))
    return ctx.tipp_aggregate_dev(pool["srs_g1"], pool["srs_g2"], a, b, c, len(idx))


def _batch(ctx, pool, idx_list):
    n = len(idx_list[0])
    flat = np.concatenate(idx_list)
    a, b, c = (ctx.to_device(x) for x in _pick(pool, flat))
    return ctx.tipp_aggregate_batch_dev(pool["srs_g1"], pool["srs_g2"], a, b, c, len(idx_list), n)


@pytest.mark.parametrize("n", [2, 4, 16, 64])
@pytest.mark.parametrize("K", [1, 3, 8])
def test_batch_equals_single_calls(ctx, pool, K, n):
    perm = np.random.default_rng(K * 1000 + n).permutation(NPOOL)
    idx_list = [perm[k * n:(k + 1) * n] for k in range(K)]
    got = _batch(ctx, pool, idx_list)
    assert len(got) == K
    for k in range(K):
        assert got[k] == _single(ctx, pool, idx_list[k]), "batch %d of %d (n = %d)" % (k, K, n)
    st = ctx.tipp_verify_aggregate_batch(pool["vsrs"], pool["vk"], [np.ascontiguousarray(pool["inputs"][i]) for i in idx_list], got)
    assert list(st) == [AGG_OK] * K


def test_repeats_and_permutations(ctx, pool):
    n = 16
    rng = np.random.default_rng(7)
    idx = [rng.permutation(NPOOL)[:n] for _ in range(4)]
    got = _batch(ctx, pool, [idx[0], idx[1], idx[0], idx[2], idx[3]])
    assert got[0] == got[2] and len({got[0], got[1], got[3], got[4]}) == 4
    order = [3, 0, 2, 1]
    perm = _batch(ctx, pool, [idx[i] for i in order])
    base = [got[0], got[1], got[3], got[4]]
    assert perm == [base[i] for i in order]
    # the host-memory entry point
    flat = np.concatenate(idx)
    a, b, c = _pick(pool, flat)
    assert ctx.tipp_aggregate_batch(pool["srs_g1"], pool["srs_g2"], a, b, c, 4) == base


def test_matches_oracle(ctx):
    n, K = 4, 2
    srs = _srs(n)
    _, proofs, _ = OS.groth16_instance(n * K)
    batches = [proofs[k * n:(k + 1) * n] for k in range(K)]
    got = aggregate_proofs_batch((srs.g_alpha_powers, srs.h_beta_powers), batches, ctx)
    for k in range(K):
        assert got[k] == O.ser_aggregate_proof(O.aggregate_proofs(srs, batches[k]))
    assert got[1] == aggregate_proofs((srs.g_alpha_powers, srs.h_beta_powers), batches[1], ctx)


def test_launch_count_does_not_grow_with_count(ctx, pool):
    n = 16
    counts = []
    for K in (2, 16):
        idx = [np.arange(k * n, (k + 1) * n) % NPOOL for k in range(K)]
        _batch(ctx, pool, idx)  # scratch sized for K
        before = ctx.launches
        _batch(ctx, pool, idx)
        counts.append(ctx.launches - before)
    assert counts[1] <= counts[0], counts


def test_argument_errors(ctx, pool):
    buf = np.zeros(1 << 20, dtype=np.uint8)
    a, b, c = pool["a"], pool["b"], pool["c"]

    def call(count=2, n=4, a=a, b=b, c=c, out=buf, cap=None, srs=None):
        plen = ctypes.c_size_t(12345)
        st = _lib.lib().ripp_tipp_aggregate_batch_dev(
            ctx.handle, _lib._p(pool["srs_g1"] if srs is None else srs), _lib._p(pool["srs_g2"]), ctypes.c_size_t(count),
            ctypes.c_size_t(n), _lib._p(a), _lib._p(b), _lib._p(c), _lib._p(out),
            ctypes.c_size_t(out.size if cap is None and out is not None else (cap or 0)), ctypes.byref(plen))
        return st, plen.value

    st, ln = call()
    assert st == _lib.RIPP_OK and ln == len(_single(ctx, pool, np.arange(4)))
    assert call(n=6)[0] == _lib.RIPP_ERR_NOT_POW2
    assert call(n=0)[0] == _lib.RIPP_ERR_NOT_POW2
    assert call(n=1)[0] == _lib.RIPP_ERR_ARG
    assert call(count=0) == (_lib.RIPP_OK, 0)
    assert call(a=None)[0] == _lib.RIPP_ERR_ARG
    assert call(c=None)[0] == _lib.RIPP_ERR_ARG
    assert call(out=None)[0] == _lib.RIPP_ERR_ARG
    assert call(srs=0)[0] == _lib.RIPP_ERR_ARG
    st, got_len = call(cap=2 * ln - 1)
    assert st == _lib.RIPP_ERR_ARG and got_len == ln
    assert call(count=(1 << 18) + 1, n=4)[0] == _lib.RIPP_ERR_ARG  # count x n over 2^20
    assert call(count=(1 << 16) + 1, n=2)[0] == _lib.RIPP_ERR_ARG  # more than 2^16 batches
    assert ctx.tipp_aggregate_batch_dev(pool["srs_g1"], pool["srs_g2"], a, b, c, 0, 4) == []


def _points(ctx, group, tag, count):
    dev = (synth.g1_points_dev if group == 1 else synth.g2_points_dev)(ctx, tag, count)
    return dev.download((count, 24 if group == 1 else 48)).copy()


def _corners(group, pts, sc, rng):
    """The corner cases of test_gpu_msm: scalars 0 / 1 / r - 1, identity bases, P and -P with equal scalars, duplicates."""
    enc, dec = (C.g1_enc, C.g1_dec) if group == 1 else (C.g2_enc, C.g2_dec)
    neg = E.g1_neg if group == 1 else E.g2_neg
    n = len(sc)
    if n >= 7:
        sc[0], sc[1], sc[2] = 0, 1, E.R - 1
        pts[3] = enc(None)
        pts[4] = pts[5]
        sc[4] = sc[5]
    if n >= 20:
        pts[12] = enc(neg(dec(pts[13])))
        sc[12] = sc[13]
    return pts, sc


@pytest.mark.parametrize("shared", [False, True])
@pytest.mark.parametrize("n", [1, 7, 1024])
@pytest.mark.parametrize("group", [1, 2])
def test_msm_batch_matches_single(ctx, group, n, shared):
    nseg = 5
    rng = np.random.default_rng(group * 100 + n)
    words = 24 if group == 1 else 48
    pts = _points(ctx, group, "mb-%d" % n, n if shared else nseg * n)
    segs_sc = []
    for s in range(nseg):
        sc = [int(x) for x in rng.integers(0, 2**62, size=n)]
        sc = [(x * 0x9E3779B97F4A7C15 + s) % E.R for x in sc]
        p = pts if shared else pts[s * n:(s + 1) * n]
        p, sc = _corners(group, p.copy(), sc, rng)
        if shared:
            pts = p
        else:
            pts[s * n:(s + 1) * n] = p
        segs_sc.append(sc)
    bases = ctx.to_device(pts)
    fr = ctx.to_device(np.concatenate([C.fr_vec_enc(sc) for sc in segs_sc]))
    out = ctx.alloc(nseg * words * 4)
    (ctx.msm_g1_batch_dev if group == 1 else ctx.msm_g2_batch_dev)(bases, 0 if shared else n, fr, n, nseg, out)
    ctx.sync()
    got = out.download((nseg, words))
    one = ctx.alloc(words * 4)
    for s in range(nseg):
        b1 = ctx.to_device(pts if shared else pts[s * n:(s + 1) * n])
        f1 = ctx.to_device(C.fr_vec_enc(segs_sc[s]))
        (ctx.msm_g1_dev if group == 1 else ctx.msm_g2_dev)(b1, f1, n, one)
        ctx.sync()
        dec = C.g1_dec if group == 1 else C.g2_dec
        assert dec(got[s]) == dec(one.download((words,))), "segment %d" % s


def test_full_size(ctx):
    """Four batches of 2^12 proofs (the seeded instance and three permutations of it) against four single calls."""
    n = 1 << 12
    t = synth.tipp_instance_dev(ctx, n)
    ha, hb, hc = t["a"].download((n, 24)), t["b"].download((n, 48)), t["c"].download((n, 24))
    rng = np.random.default_rng(11)
    perms = [np.arange(n)] + [rng.permutation(n) for _ in range(3)]
    got = ctx.tipp_aggregate_batch(t["srs_g1"], t["srs_g2"], np.concatenate([ha[p] for p in perms]),
                                   np.concatenate([hb[p] for p in perms]), np.concatenate([hc[p] for p in perms]), 4)
    for k, p in enumerate(perms):
        a, b, c = ctx.to_device(ha[p]), ctx.to_device(hb[p]), ctx.to_device(hc[p])
        assert got[k] == ctx.tipp_aggregate_dev(t["srs_g1"], t["srs_g2"], a, b, c, n), "batch %d" % k
