"""The algebra of the batched polynomial-commitment verifier (ripp_b200/csrc/pc_verify_batch.cuh), restated on the
oracle: every check of the trusted and transparent verify as a product of at most three pairings against a target, a
G1 identity or an Fr equation, with the final keys of the transparent kind built from exponents by the bit rule of
pc::key_exponent.  These are group identities, so they must decide exactly as the oracle's verify does; among the cases
is a transparent opening with a0 = O and b0 != the SSM scalar, which verify accepts and a rewrite of the two G1
identities into `b0 == ssm` would reject."""
import pytest

from oracle import bls12_381 as E
from oracle import poly_commit as OPC
from oracle import protocols as O
from oracle import synth as OS
from oracle.encoding import blake2b, ser_fr, ser_g2

R = E.R
ALPHA, BETA = OS.scalar("pcv-oracle-alpha", 0), OS.scalar("pcv-oracle-beta", 0)


def _eq(pairs, target=E.F12_ONE):
    acc = E.F12_ONE
    for p, q in pairs:
        acc = E.gt_mul(acc, E.pairing(p, q))
    return acc == target


def _mul(p, s):
    return E.g1_mul(p, s % R)


def _add(*pts):
    acc = None
    for p in pts:
        acc = E.g1_add(acc, p)
    return acc


def _key(points, transcript, factor, add, mul):
    """factor * sum_i e_i points[i], e_i = prod over the bits j set in i of transcript[j]^-1 (pc::key_exponent)."""
    tinv = [E.fr_inv(x) for x in transcript]
    acc = None
    for i, p in enumerate(points):
        e = factor
        for j in range(len(tinv)):
            if i >> j & 1:
                e = e * tinv[j] % R
        acc = add(acc, mul(p, e))
    return acc


def trusted_checks(vs, com, point, evaluation, proof):
    """-> {name: bool}: the checks of one trusted opening as the batched verifier states them."""
    g, h, g_beta, h_alpha = vs["g"], vs["h"], vs["g_beta"], vs["h_alpha"]
    x, y = point
    ip, ye, pik = proof["ip_proof"], proof["y_eval_comm"], proof["kzg_proof"]
    gipa = OPC._ipa().gipa
    if not ip.gipa_proof.r_commitment_steps:
        return {"rounds": False}
    fold, t = gipa.compute_recursive_challenges((com, x, [ye]), ip.gipa_proof)
    tinv = [E.fr_inv(c) for c in t]
    ck, pi = ip.final_ck, ip.final_ck_proof
    z = O._kzg_challenge(blake2b, ser_fr(t[0]) + ser_g2(ck))
    fa = O.polynomial_evaluation_product_form_from_transcript(tinv, z, 1)
    a0 = ip.gipa_proof.r_base[0]
    return {
        "kzg_final_key": _eq([(g, ck), (_mul(g, -fa), h), (_add(_mul(g, z), E.g1_neg(g_beta)), pi)]),
        "base": _eq([(a0, ck)], fold[0]),
        "kzg_at_y": _eq([(_add(ye, _mul(g, -evaluation), _mul(pik, y)), h), (E.g1_neg(pik), h_alpha)]),
        "g1_identity": _add(fold[2][0], _mul(a0, -O._ssm_final_scalar(t, x))) is None,
    }


def transparent_checks(ck, com, point, evaluation, proof):
    first, second = ck
    x, y = point
    p2, ye, p1 = proof["second_tier_ip_proof"], proof["y_eval_comm"], proof["first_tier_ip_proof"]
    out = {"rounds": len(p2.r_commitment_steps) == len(second).bit_length() - 1
           and len(p1.r_commitment_steps) == len(first).bit_length() - 1}
    if not out["rounds"]:
        return out
    fold2, t2 = OPC._second_tier().gipa.compute_recursive_challenges((com, 0, [ye]), p2)
    a0, b0 = p2.r_base
    ck2 = _key(second, t2, 1, E.g2_add, E.g2_mul)
    out["base"] = _eq([(a0, ck2)], fold2[0])
    out["placeholder_2"] = fold2[1] % R == 0
    out["g1_b0"] = _add(fold2[2][0], _mul(a0, -b0)) is None
    out["g1_ssm"] = _add(fold2[2][0], _mul(a0, -O._ssm_final_scalar(t2, x))) is None
    fold1, t1 = OPC._first_tier().gipa.compute_recursive_challenges((ye, 0, [evaluation]), p1)
    a1, b1 = p1.r_base
    out["g1_first_tier"] = _add(fold1[0], E.g1_neg(_key(first, t1, a1, E.g1_add, E.g1_mul))) is None
    out["placeholder_1"] = fold1[1] % R == 0
    out["eval_b0"] = fold1[2][0] % R == a1 * b1 % R
    out["eval_ssm"] = fold1[2][0] % R == a1 * O._ssm_final_scalar(t1, y) % R
    return out


def _copy_gipa(p, steps=None, base=None):
    return O.GIPAProof(list(p.r_commitment_steps) if steps is None else steps, p.r_base if base is None else base)


def _tamper_round(p):
    steps = list(p.r_commitment_steps)
    c1, c2 = steps[0]
    steps[0] = ((E.gt_mul(c1[0], c1[0]),) + tuple(c1[1:]), c2)
    return _copy_gipa(p, steps)


def test_trusted_identities_decide_as_verify():
    n, m = 2, 2
    srs = OPC.BivariatePolynomialCommitment.setup(n - 1, m - 1, ALPHA, BETA)
    vs = srs[0].get_verifier_key()
    polys = [[OS.scalar("pcv-t", i * m + j) for j in range(m)] for i in range(n)]
    com, y_coms = OPC.BivariatePolynomialCommitment.commit(srs, polys)
    point = (OS.scalar("pcv-x", 0), OS.scalar("pcv-y", 0))
    proof = OPC.BivariatePolynomialCommitment.open(srs, polys, y_coms, point)
    ev = OPC.bivariate_evaluate(polys, point)
    ip = proof["ip_proof"]
    cases = [
        ("valid", point, ev, proof),
        ("wrong eval", point, ev + 1, proof),
        ("wrong point", (point[0], point[1] + 1), ev, proof),
        ("round commitment", point, ev, dict(proof, ip_proof=O.TIPAWithSSMProof(_tamper_round(ip.gipa_proof), ip.final_ck,
                                                                              ip.final_ck_proof))),
        ("final key", point, ev, dict(proof, ip_proof=O.TIPAWithSSMProof(ip.gipa_proof, E.g2_add(ip.final_ck, E.G2_GEN),
                                                                       ip.final_ck_proof))),
        ("kzg proof", point, ev, dict(proof, kzg_proof=E.g1_add(proof["kzg_proof"], E.G1_GEN))),
    ]
    for name, pt, e, pf in cases:
        want = OPC.BivariatePolynomialCommitment.verify(vs, com, pt, e % R, pf)
        got = trusted_checks(vs, com, pt, e % R, pf)
        assert all(got.values()) == want, (name, got)
        assert want == (name == "valid"), name


@pytest.mark.parametrize("zero", [False, True])
def test_transparent_identities_decide_as_verify(zero):
    n, m = 2, 2
    ck = (OS.g1_points("pcv-ck1", m), OS.g2_points("pcv-ck2", n))
    polys = [[0 if zero else OS.scalar("pcv-p", i * m + j) for j in range(m)] for i in range(n)]
    com, y_coms = OPC.TransparentBivariatePolynomialCommitment.commit(ck, polys)
    point = (OS.scalar("pcv-x", 1), OS.scalar("pcv-y", 1))
    proof = OPC.TransparentBivariatePolynomialCommitment.open(ck, polys, y_coms, point)
    ev = OPC.bivariate_evaluate(polys, point)
    p2, p1 = proof["second_tier_ip_proof"], proof["first_tier_ip_proof"]
    a0, b0 = p2.r_base
    changed_b0 = dict(proof, second_tier_ip_proof=_copy_gipa(p2, base=(a0, (b0 + 1) % R)))
    cases = [("valid", point, ev, proof, True), ("b0 changed", point, ev, changed_b0, zero)]
    if not zero:
        steps = list(p1.r_commitment_steps)
        c1, c2 = steps[0]
        steps[0] = ((c1[0], 5, c1[2]), c2)
        a1, b1 = p1.r_base
        cases += [
            ("wrong eval", point, ev + 1, proof, False),
            ("wrong point", (point[0] + 1, point[1]), ev, proof, False),
            ("round commitment", point, ev, dict(proof, second_tier_ip_proof=_tamper_round(p2)), False),
            ("y_eval_comm", point, ev, dict(proof, y_eval_comm=E.g1_add(proof["y_eval_comm"], E.G1_GEN)), False),
            ("first-tier placeholder", point, ev, dict(proof, first_tier_ip_proof=_copy_gipa(p1, steps)), False),
            ("first-tier b0", point, ev, dict(proof, first_tier_ip_proof=_copy_gipa(p1, base=(a1, (b1 + 1) % R))), False),
        ]
    else:
        assert a0 is None  # a0 = O: the two G1 identities coincide, and b0 is not checked
    for name, pt, e, pf, accept in cases:
        want = OPC.TransparentBivariatePolynomialCommitment.verify(ck, com, pt, e % R, pf)
        got = transparent_checks(ck, com, pt, e % R, pf)
        assert all(got.values()) == want == accept, (name, got)
