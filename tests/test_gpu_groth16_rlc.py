"""Groth16 verification by random linear combination on the GPU (ripp_groth16_verify_rlc_dev / _serialized): verdicts
and statuses equal the per-proof entry points' and the oracle's, and the number of proofs re-checked one by one equals
the oracle's count exactly (oracle/groth16_rlc.py) -- a wrong combination would only make segments fail, and the
fallback would still give the right verdicts, so the count is what shows the combination is right.  The segment size
is a per-process switch: the forced sizes (one proof, partial segments, one segment for everything) run in
subprocesses."""
import importlib.util
import os
import subprocess
import sys

import numpy as np
import pytest

from oracle import groth16 as G
from oracle import groth16_rlc as Q
from oracle import serde as S
from oracle import serde_cases as SC
from ripp_b200 import _lib
from ripp_b200 import groth16 as R

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEG = int(os.environ.get("RIPP_B200_G16_RLC_SEG", "58"))  # the library's default segment size (include/ripp_b200.h)
SEED = bytes(range(32))

# the batch builders of the per-proof entry points' tests
_spec = importlib.util.spec_from_file_location("_g16_cases", os.path.join(ROOT, "tests", "test_gpu_groth16.py"))
T = importlib.util.module_from_spec(_spec)
_spec.loader.exec_module(T)


def _expected(seed, vk, ic, proofs, inputs, members, truth):
    return Q.rlc_expected(seed, members, SEG, lambda r, idx: Q.rlc_segment_exponent(vk, ic, proofs, inputs, r, idx), truth)


@pytest.fixture(scope="module")
def mixed():
    out = {}
    for m in (0, 1, 5):
        vk, ic, proofs, inputs, kinds = G.groth16_mixed_scalars(m)
        vkp, pts = G.groth16_points(vk, ic, proofs)
        pvk = G.prepare_verifying_key(vkp)
        out[m] = (vk, ic, proofs, inputs, vkp, pts, [G.verify_proof(pvk, p, x) for p, x in zip(pts, inputs)])
    return out


@pytest.mark.parametrize("m", [0, 1, 5])
def test_verdicts_and_rechecks_match_oracle(ctx, mixed, m):
    vk, ic, proofs, inputs, vkp, pts, want = mixed[m]
    pvk = R.prepare_verifying_key(vkp, ctx)
    for n in (len(pts), 1, 2, 37, 40):
        idx = list(range(n)) if n == len(pts) else [(7 * i + 3) % len(pts) for i in range(n)]
        sub_p, sub_x, sub_w = [proofs[i] for i in idx], [inputs[i] for i in idx], [want[i] for i in idx]
        got, nre = R.verify_proofs_rlc(pvk, sub_x, [pts[i] for i in idx], seed=SEED)
        assert got == sub_w == R.verify_proofs(pvk, sub_x, [pts[i] for i in idx]), n
        exp, exp_nre = _expected(SEED, vk, ic, sub_p, sub_x, [True] * n, sub_w)
        assert exp == sub_w and nre == exp_nre, (n, nre, exp_nre)
        if all(sub_w):
            assert nre == 0


@pytest.mark.parametrize("compressed", [True, False])
@pytest.mark.parametrize("m", [0, 1, 5])
def test_serialized_statuses_match_per_proof_entry(ctx, mixed, m, compressed):
    vk, ic, proofs, inputs, vkp, pts, _ = mixed[m]
    pvk = R.prepare_verifying_key(vkp, ctx)
    data, rows = T._serialized_batch(pts, inputs, compressed, seed=m)
    xb, n = T._xbytes(rows), len(pts)
    want, nv_want = ctx.groth16_verify_serialized(pvk.buf, m, xb, data, n, compressed)
    st, nv, nre = ctx.groth16_verify_rlc_serialized(pvk.buf, m, xb, data, n, compressed, SEED)
    assert st.tolist() == want.tolist() and nv == nv_want
    members = [int(w) in (S.OK, G.REJECTED) for w in want]
    assert not all(members)
    _, exp_nre = _expected(SEED, vk, ic, proofs, rows, members, [int(w) == S.OK for w in want])
    assert nre == exp_nre
    assert R.verify_proofs_serialized_rlc(pvk, xb, data, compressed, seed=SEED)[0].tolist() == want.tolist()
    # a segment whose members are all excluded: three proofs with bad encodings
    bad = [i for i, mem in enumerate(members) if not mem][:3]
    rec = 192 if compressed else 384
    d3 = b"".join(data[i * rec : (i + 1) * rec] for i in bad)
    x3 = T._xbytes([rows[i] for i in bad])
    st, nv, nre = ctx.groth16_verify_rlc_serialized(pvk.buf, m, x3, d3, len(bad), compressed, SEED)
    assert st.tolist() == [int(want[i]) for i in bad] and nv == 0 and nre == 0


def test_refuses_null_seed_and_bad_lengths(ctx, mixed):
    vk, ic, proofs, inputs, vkp, pts, _ = mixed[1]
    pvk = R.prepare_verifying_key(vkp, ctx)
    data, xb, n = T._record(pts[0], True) + T._record(pts[1], True), T._xbytes(inputs[:2]), 2
    for d, x, cnt, sd in ((data, xb, n, None), (data[:-1], xb, n, SEED), (data + b"\x00", xb, n, SEED), (data, xb[:-1], n, SEED),
                          (data, xb + b"\x00" * 32, n, SEED), (data, xb, n + 1, SEED), (data, xb, 1, SEED)):
        with pytest.raises(_lib.RippError) as e:
            ctx.groth16_verify_rlc_serialized(pvk.buf, 1, x, d, cnt, True, sd)
        assert e.value.status == _lib.RIPP_ERR_ARG, (len(d), len(x), cnt, sd)
    a, b, c, x = R._upload(pvk, inputs[:2], pts[:2])
    out = ctx.alloc(2)
    with pytest.raises(_lib.RippError) as e:
        ctx.groth16_verify_rlc_dev(pvk.buf, 1, x, a, b, c, 2, None, out)
    assert e.value.status == _lib.RIPP_ERR_ARG
    with pytest.raises(ValueError):
        R.verify_proofs_rlc(pvk, inputs[:2], pts[:2], seed=b"short")
    assert R.verify_proofs_rlc(pvk, [], []) == ([], 0)
    assert ctx.groth16_verify_rlc_serialized(pvk.buf, 1, b"", b"", 0, True, SEED)[1:] == (0, 0)


def test_seeds(ctx, mixed):
    vk, ic, proofs, inputs, vkp, pts, want = mixed[5]
    pvk = R.prepare_verifying_key(vkp, ctx)
    s2 = bytes(range(100, 132))
    g1, n1 = R.verify_proofs_rlc(pvk, inputs, pts, seed=SEED)
    g2, n2 = R.verify_proofs_rlc(pvk, inputs, pts, seed=s2)
    g3, n3 = R.verify_proofs_rlc(pvk, inputs, pts, seed=SEED)
    g4, _ = R.verify_proofs_rlc(pvk, inputs, pts)
    assert g1 == g2 == g3 == g4 == want and n1 == n3
    assert n2 == _expected(s2, vk, ic, proofs, inputs, [True] * len(pts), want)[1]


# ---- large batches against the exponent-space truth ---------------------------------------------------------------
def _rlc_dev(ctx, vk_words, m, x, a, b, c, n, seed):
    pvk = ctx.alloc(ctx.groth16_pvk_bytes(m))
    ctx.groth16_prepare_vk_dev(vk_words, m, pvk)
    out = ctx.alloc(n)
    nre = ctx.groth16_verify_rlc_dev(pvk, m, x, a, b, c, n, seed, out)
    return pvk, out.download(n, dtype=np.uint8), nre


@pytest.mark.parametrize("lg,nfalse", [(12, 41), (16, 0), (16, 5)])
def test_large(ctx, lg, nfalse):
    n, m = 1 << lg, 5
    vk_words, a, b, c, x, inputs, truth, pos = T._large(ctx, n, m, nfalse, seed=lg + nfalse)
    assert truth.count(False) == nfalse
    # the exponents again (as T._large draws them) for the expected re-check count
    sc, proofs, _ = T.OS.groth16_instance_scalars(n, m, lg + nfalse)
    proofs = list(proofs)
    ref_inputs = [list(xr) for xr in T.OS.groth16_instance_scalars(n, m, lg + nfalse)[2]]
    _replay_tamper(sc["vk"], sc["ic"], proofs, ref_inputs, pos, lg + nfalse, n, nfalse)
    assert ref_inputs == inputs
    exp, exp_nre = _expected(SEED, sc["vk"], sc["ic"], proofs, inputs, [True] * n, truth)
    pvk, got, nre = _rlc_dev(ctx, vk_words, m, x, a, b, c, n, SEED)
    assert got.tolist() == [int(t) for t in truth] and nre == exp_nre
    if nfalse == 0:
        assert nre == 0
    if lg == 12:
        data = SC.proof_records(a.download((n, 24)), b.download((n, 48)), c.download((n, 24)), True)
        st, nv, nre = ctx.groth16_verify_rlc_serialized(pvk, m, T._xbytes(inputs), data, n, True, SEED)
        assert st.tolist() == [S.OK if t else G.REJECTED for t in truth] and nv == n - nfalse and nre == exp_nre


def _replay_tamper(vk, ic, proofs, inputs, pos, seed, n, nfalse):
    """T._large's tampering of the exponents, replayed (it returns the points, not the exponents)."""
    import random

    rng = random.Random(seed)
    p = rng.sample(range(n), nfalse)
    k = 0
    while k < len(p):
        kind = G.GROTH16_TAMPER[k % 4]
        if kind == "b_swapped" and k + 1 < len(p):
            G.groth16_tamper(vk, ic, proofs, inputs, kind, p[k], p[k + 1])
            k += 2
            continue
        G.groth16_tamper(vk, ic, proofs, inputs, "c_plus_g" if kind == "b_swapped" else kind, p[k])
        k += 1
    assert sorted(p) == pos


# ---- forced segment sizes -----------------------------------------------------------------------------------------
@pytest.mark.parametrize("seg", ["1", "7", "100000"])
def test_forced_segment_sizes(seg):
    if "RIPP_B200_G16_RLC_SEG" in os.environ:
        pytest.skip("already running with a forced segment size")
    sel = ["tests/test_gpu_groth16_rlc.py::test_verdicts_and_rechecks_match_oracle",
           "tests/test_gpu_groth16_rlc.py::test_serialized_statuses_match_per_proof_entry",
           "tests/test_gpu_groth16_rlc.py::test_seeds"]
    if seg == "7":
        sel.append("tests/test_gpu_groth16_rlc.py::test_large[12-41]")
    r = subprocess.run([sys.executable, "-m", "pytest", "-q", "-x", "-m", "gpu"] + sel, cwd=ROOT,
                       env=dict(os.environ, RIPP_B200_G16_RLC_SEG=seg), capture_output=True, text=True, timeout=1500)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
