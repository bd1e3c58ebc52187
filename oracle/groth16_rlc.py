"""ORACLE (test infrastructure, NOT product code) -- Groth16 batch verification by random linear combination
(ripp_groth16_verify_rlc_dev / _serialized).  ark-groth16 0.4 has no batch verifier, so these functions state the
library's own rule: segments of s consecutive proofs, ChaCha20 scalars normalised to sum to one per segment, one
combined pairing check per segment, and the per-proof verdict (oracle/groth16.py) for the members of failing segments.
"""
from . import bls12_381 as E
from . import encoding as enc
from .groth16 import prepare_inputs


def rlc_scalars(seed, members, s):
    """The scalars of the segment checks: r_i = the i-th 16-byte little-endian chunk of the ChaCha20 keystream keyed by
    the 32-byte seed (four per 64-byte block), 0 for non-members; in each segment of s consecutive proofs the last
    member takes 1 - (the other members' sum) mod r instead."""
    n = len(members)
    ks = b"".join(enc.chacha20_block(seed, b) for b in range((n + 3) // 4))
    r = [int.from_bytes(ks[16 * i : 16 * i + 16], "little") if members[i] else 0 for i in range(n)]
    for lo in range(0, n, s):
        idx = [i for i in range(lo, min(n, lo + s)) if members[i]]
        if idx:
            r[idx[-1]] = (1 - sum(r[i] for i in idx[:-1])) % E.R
    return r


def rlc_segment_check(pvk, proofs, inputs, r, idx):
    """One segment's check over the pairing: final_exp(prod_i ML(r_i A_i, B_i) ML(P_s, -gamma) ML(C_s, -delta)) ==
    e(alpha, beta) with P_s = prepare_inputs(sigma_s), sigma_sj = sum_i r_i x_ij, C_s = sum_i r_i C_i (i in idx)."""
    m = len(pvk["gamma_abc_g1"]) - 1
    sigma = [sum(r[i] * inputs[i][j] for i in idx) % E.R for j in range(m)]
    cs = None
    for i in idx:
        cs = E.g1_add(cs, E.g1_mul(proofs[i][2], r[i]))
    g1 = [E.g1_mul(proofs[i][0], r[i]) for i in idx] + [prepare_inputs(pvk, sigma), cs]
    g2 = [proofs[i][1] for i in idx] + [pvk["gamma_g2_neg_pc"], pvk["delta_g2_neg_pc"]]
    return E.multi_pairing(g1, g2) == pvk["alpha_g1_beta_g2"]


def rlc_segment_exponent(vk, ic, proofs, inputs, r, idx):
    """The same check on trapdoor-simulated proofs (exponents, as groth16_exponent_verdict): sum_i r_i a_i b_i ==
    alpha beta + gamma (ic_0 + sum_j sigma_j ic_j) + delta sum_i r_i c_i (mod r)."""
    R = E.R
    m = len(ic) - 1
    sigma = [sum(r[i] * inputs[i][j] for i in idx) % R for j in range(m)]
    icx = (ic[0] + sum(sj * icj for sj, icj in zip(sigma, ic[1:]))) % R
    lhs = sum(r[i] * proofs[i][0] * proofs[i][1] for i in idx)
    return (lhs - vk["alpha"] * vk["beta"] - vk["gamma"] * icx - vk["delta"] * sum(r[i] * proofs[i][2] for i in idx)) % R == 0


def rlc_expected(seed, members, s, segment_ok, truth):
    """Verdicts of the random-linear-combination entry points and the exact number of proofs they re-check:
    segment_ok(r, idx) decides a segment (rlc_segment_check / rlc_segment_exponent with the batch bound), truth[i] is
    the per-proof verdict.  -> (verdicts, n_rechecked); None for non-members, which keep their status."""
    n = len(members)
    r = rlc_scalars(seed, members, s)
    out, rechecked = [None] * n, 0
    for lo in range(0, n, s):
        idx = [i for i in range(lo, min(n, lo + s)) if members[i]]
        if not idx:
            continue
        ok = segment_ok(r, idx)
        for i in idx:
            out[i] = True if ok else truth[i]
        rechecked += 0 if ok else len(idx)
    return out, rechecked
