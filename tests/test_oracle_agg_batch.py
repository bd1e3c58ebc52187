"""The algebra of the batched aggregate verifier (ripp_b200/csrc/verify_batch.cuh), restated on the oracle: every check
of verify_aggregate_proof rewritten as a product of at most three pairings against a target (scalars moved to the G1
side by bilinearity) or as a G1 identity.  These rewrites are group identities, so they must decide exactly as
verify_aggregate_proof does; pinned here before any GPU run."""
import pytest

from oracle import bls12_381 as E
from oracle import protocols as O
from oracle import synth as OS
from oracle.encoding import blake2b, ser_fr, ser_g1, ser_g2

R = E.R


def _eq(pairs, target=E.F12_ONE):
    acc = E.F12_ONE
    for p, q in pairs:
        acc = E.gt_mul(acc, E.pairing(p, q))
    return acc == target


def _mul(p, s):
    return E.g1_mul(p, s % R)


def batch_checks(vs, vk, inputs, agg):
    """-> {name: bool}, the checks of one aggregate as the batched verifier states them."""
    g, h, g_beta, h_alpha = vs["g"], vs["h"], vs["g_beta"], vs["h_alpha"]
    r = O._agg_challenge(blake2b, agg.com_a, agg.com_b, agg.com_c)
    out = {}
    # AB proof: GT folds of com_a, com_b, ip_ab; KZG openings of both final keys; base checks
    tab, pab = O._tipp_ab(blake2b, None), agg.tipa_proof_ab
    fold, t = tab.gipa.compute_recursive_challenges((agg.com_a, agg.com_b, [agg.ip_ab]), pab.gipa_proof)
    tinv = [E.fr_inv(x) for x in t]
    (ck_a, ck_b), (pi_a, pi_b) = pab.final_ck, pab.final_ck_proof
    z = O._kzg_challenge(blake2b, ser_fr(t[0]) + ser_g2(ck_a) + ser_g1(ck_b))
    fa = O.polynomial_evaluation_product_form_from_transcript(tinv, z, E.fr_inv(r))
    fb = O.polynomial_evaluation_product_form_from_transcript(t, z, 1)
    out["kzg_ab_g2"] = _eq([(g, ck_a), (_mul(g, -fa), h), (E.g1_add(_mul(g, z), E.g1_neg(g_beta)), pi_a)])
    out["kzg_ab_g1"] = _eq([(E.g1_add(E.g1_add(ck_b, _mul(g, -fb)), _mul(pi_b, z)), h), (E.g1_neg(pi_b), h_alpha)])
    assert out["kzg_ab_g2"] == O.verify_commitment_key_g2_kzg_opening(vs, ck_a, pi_a, tinv, E.fr_inv(r), z)
    assert out["kzg_ab_g1"] == O.verify_commitment_key_g1_kzg_opening(vs, ck_b, pi_b, t, 1, z)
    a0, b0 = pab.gipa_proof.r_base
    out["base_com_a"] = _eq([(a0, ck_a)], fold[0])
    out["base_com_b"] = _eq([(ck_b, b0)], fold[1])
    out["base_ip_ab"] = _eq([(a0, b0)], fold[2][0])
    # C proof: GT fold of com_c, KZG opening of the final G2 key, base check, and the G1 identity of agg_c's fold
    tc, pc = O._tipp_c(blake2b, None), agg.tipa_proof_c
    fold_c, t = tc.gipa.compute_recursive_challenges((agg.com_c, r, [agg.agg_c]), pc.gipa_proof)
    tinv = [E.fr_inv(x) for x in t]
    z = O._kzg_challenge(blake2b, ser_fr(t[0]) + ser_g2(pc.final_ck))
    fa = O.polynomial_evaluation_product_form_from_transcript(tinv, z, 1)
    out["kzg_c_g2"] = _eq([(g, pc.final_ck), (_mul(g, -fa), h), (E.g1_add(_mul(g, z), E.g1_neg(g_beta)), pc.final_ck_proof)])
    assert out["kzg_c_g2"] == O.verify_commitment_key_g2_kzg_opening(vs, pc.final_ck, pc.final_ck_proof, tinv, 1, z)
    a0c = pc.gipa_proof.r_base[0]
    out["base_com_c"] = _eq([(a0c, pc.final_ck)], fold_c[0])
    out["g1_identity"] = E.g1_add(fold_c[2][0], _mul(a0c, -O._ssm_final_scalar(t, r))) is None
    # the Groth16 product equation against ip_ab
    n = len(inputs)
    r_sum = (pow(r, n, R) - 1) * E.fr_inv((r - 1) % R) % R
    r_vec = O.structured_scalar_power(n, r)
    g_ic = _mul(vk["gamma_abc_g1"][0], r_sum)
    for j, b in enumerate(vk["gamma_abc_g1"][1:]):
        g_ic = E.g1_add(g_ic, _mul(b, sum(row[j] * x for row, x in zip(inputs, r_vec))))
    out["ppe"] = _eq([(_mul(vk["alpha_g1"], r_sum), vk["beta_g2"]), (g_ic, vk["gamma_g2"]), (agg.agg_c, vk["delta_g2"])], agg.ip_ab)
    return out


@pytest.mark.parametrize("n", [2, 4])
def test_rewritten_checks_decide_as_verify_aggregate_proof(n):
    srs = O.tipa_setup(n, OS.scalar("srs-alpha", 0), OS.scalar("srs-beta", 0))
    vs = srs.get_verifier_key()
    vk, proofs, inputs = OS.groth16_instance(n)
    agg = O.aggregate_proofs(srs, proofs)
    bad_inputs = [list(x) for x in inputs]
    bad_inputs[n - 1][1] = (bad_inputs[n - 1][1] + 1) % R
    bad_kzg = O.AggregateProof(**dict(agg.__dict__))
    ab = agg.tipa_proof_ab
    bad_kzg.tipa_proof_ab = O.TIPAProof(ab.gipa_proof, ab.final_ck, (E.g2_add(ab.final_ck_proof[0], E.G2_GEN), ab.final_ck_proof[1]))
    bad_ip = O.AggregateProof(**dict(agg.__dict__))
    bad_ip.ip_ab = E.gt_mul(agg.ip_ab, E.pairing(E.G1_GEN, E.G2_GEN))
    cases = {"honest": (inputs, agg), "input": (bad_inputs, agg), "kzg": (inputs, bad_kzg), "ip_ab": (inputs, bad_ip)}
    failing = {"honest": set(), "input": {"ppe"}, "kzg": {"kzg_ab_g2"}, "ip_ab": {"base_ip_ab", "ppe"}}
    for name, (x, a) in cases.items():
        checks = batch_checks(vs, vk, x, a)
        assert {k for k, v in checks.items() if not v} == failing[name], name
        assert all(checks.values()) == O.verify_aggregate_proof(vs, vk, x, a), name
