"""ORACLE (test infrastructure, NOT product code) -- ark-groth16 0.4 verification over the pure-Python pairing.

PARITY UNPINNED: the semantics are recalled, not read from the crate (it is not vendored here, as SURVEY.md App. A
recalls other arkworks behaviour); tools/ark_golden dumps ark-groth16's own verdicts for tests/test_gpu_groth16.py.
  prepare_verifying_key: alpha_g1_beta_g2 = e(alpha, beta), gamma_g2_neg_pc = -gamma, delta_g2_neg_pc = -delta
  prepare_inputs(pvk, x) = IC_0 + sum_j x_j IC_j, an error unless len(x) + 1 == len(gamma_abc_g1)
  verify_proof: final_exp(multi_miller_loop([A, P, C], [B, -gamma, -delta])) == e(alpha, beta)
Points are affine tuples, None for the identity; vk is the dict of oracle.synth.groth16_instance.
"""
from . import bls12_381 as E
from . import serde as S
from . import synth

# statuses of a serialized (proof record, inputs) pair: 0..4 the point decode status of A, B or C (the first that
# fails), then a public input >= r, then a false equation
INPUT_NONCANONICAL, REJECTED = 5, 6


def prepare_verifying_key(vk):
    return {
        "alpha_g1_beta_g2": E.pairing(vk["alpha_g1"], vk["beta_g2"]),
        "gamma_g2_neg_pc": E.g2_neg(vk["gamma_g2"]),
        "delta_g2_neg_pc": E.g2_neg(vk["delta_g2"]),
        "gamma_abc_g1": list(vk["gamma_abc_g1"]),
    }


def prepare_inputs(pvk, x):
    ic = pvk["gamma_abc_g1"]
    if len(x) + 1 != len(ic):
        raise ValueError("MalformedVerifyingKey: %d public inputs for %d gamma_abc_g1 points" % (len(x), len(ic)))
    acc = ic[0]
    for xj, icj in zip(x, ic[1:]):
        acc = E.g1_add(acc, E.g1_mul(icj, xj))
    return acc


def verify_proof(pvk, proof, x):
    a, b, c = proof
    p = prepare_inputs(pvk, x)
    f = E.multi_pairing([a, p, c], [b, pvk["gamma_g2_neg_pc"], pvk["delta_g2_neg_pc"]])
    return f == pvk["alpha_g1_beta_g2"]


def decode_inputs(data, m):
    """m ark-serialize Fr (32 bytes little-endian each) -> (ints, canonical?)"""
    if len(data) != 32 * m:
        raise ValueError("expected %d bytes, got %d" % (32 * m, len(data)))
    x = [int.from_bytes(data[32 * j : 32 * j + 32], "little") for j in range(m)]
    return x, all(v < E.R for v in x)


def status_serialized(pvk, record, inputs, compressed):
    """Expected status of one ark-groth16 Proof record (serialize_compressed / _uncompressed) with its inputs' bytes."""
    g1b = 48 if compressed else 96
    parts = ((S.de_g1, record[:g1b]), (S.de_g2, record[g1b : 3 * g1b]), (S.de_g1, record[3 * g1b :]))
    pts = []
    for de, b in parts:
        pt, st = de(b, compressed)
        if st != S.OK:
            return st
        pts.append(pt)
    x, canonical = decode_inputs(inputs, len(pvk["gamma_abc_g1"]) - 1)
    if not canonical:
        return INPUT_NONCANONICAL
    return S.OK if verify_proof(pvk, tuple(pts), x) else REJECTED


def ser_vk_compressed(vk):
    """ark-groth16 VerifyingKey::serialize_compressed: alpha_g1, beta_g2, gamma_g2, delta_g2, gamma_abc_g1 (u64 LE
    length, then the points)."""
    ic = vk["gamma_abc_g1"]
    return (S.ser_g1_compressed(vk["alpha_g1"]) + S.ser_g2_compressed(vk["beta_g2"]) + S.ser_g2_compressed(vk["gamma_g2"])
            + S.ser_g2_compressed(vk["delta_g2"]) + len(ic).to_bytes(8, "little") + b"".join(S.ser_g1_compressed(p) for p in ic))


def golden_case_lines():
    """tests/golden/groth16_cases.txt: the m = 1 mixed batch below as ark-groth16 would read it --
    `groth16_vk <hex>`, then `groth16_case_<i> <Proof compressed hex> <inputs hex>` (the verdicts tools/ark_golden dumps)."""
    vk, ic, proofs, inputs, kinds = groth16_mixed_scalars(1)
    vkp, pts = groth16_points(vk, ic, proofs)
    lines = ["groth16_vk %s" % ser_vk_compressed(vkp).hex()]
    for i, (p, x) in enumerate(zip(pts, inputs)):
        rec = S.ser_g1_compressed(p[0]) + S.ser_g2_compressed(p[1]) + S.ser_g1_compressed(p[2])
        lines.append("groth16_case_%d %s %s" % (i, rec.hex(), b"".join(v.to_bytes(32, "little") for v in x).hex()))
    return "\n".join(lines) + "\n"


# ---- truth in exponent space, tampered and edge-case proofs (trapdoor-simulated as oracle/synth.py makes them) ----
def groth16_exponent_verdict(vk, ic, proof, x):
    """ark-groth16 verify_proof on trapdoor-simulated proofs (known discrete logs; vk, ic as groth16_instance_scalars):
    valid iff a b == alpha beta + gamma (ic_0 + sum_j ic_j x_j) + delta c (mod r).  Length mismatch raises."""
    if len(x) + 1 != len(ic):
        raise ValueError("MalformedVerifyingKey: %d public inputs for %d gamma_abc_g1 points" % (len(x), len(ic)))
    R = E.R
    a, b, c = proof
    icx = (ic[0] + sum(xj * icj for xj, icj in zip(x, ic[1:]))) % R
    return (a * b - vk["alpha"] * vk["beta"] - vk["gamma"] * icx - vk["delta"] * c) % R == 0


def _groth16_c(vk, ic, a, b, x):
    icx = (ic[0] + sum(xj * icj for xj, icj in zip(x, ic[1:]))) % E.R
    return (a * b - vk["alpha"] * vk["beta"] - vk["gamma"] * icx) * pow(vk["delta"], -1, E.R) % E.R


GROTH16_TAMPER = ("c_plus_g", "input_changed", "b_swapped", "a_scaled")
GROTH16_EDGE = ("p_identity", "c_identity", "a_identity", "b_identity", "input_r_minus_1")


def groth16_tamper(vk, ic, proofs, inputs, kind, i, j=None):
    """Apply one tamper class to proof i in place, keeping every discrete log known (all of them make it false):
    c_plus_g C + G; input_changed x_i0 + 1 (needs an input); b_swapped B_i <-> B_j (both false unless b_i = b_j);
    a_scaled 2 A."""
    a, b, c = proofs[i]
    if kind == "c_plus_g":
        proofs[i] = (a, b, (c + 1) % E.R)
    elif kind == "input_changed":
        inputs[i] = [(inputs[i][0] + 1) % E.R] + list(inputs[i][1:])
    elif kind == "b_swapped":
        aj, bj, cj = proofs[j]
        proofs[i], proofs[j] = (a, bj, c), (aj, b, cj)
    elif kind == "a_scaled":
        proofs[i] = (2 * a % E.R, b, c)
    else:
        raise ValueError(kind)


def groth16_edge(vk, ic, kind, seed=0):
    """One proof (a, b, c) with its inputs for an edge class the kernels must mask: p_identity (valid, P = O: x_1
    solved so that ic_0 + sum ic_j x_j = 0; needs an input), c_identity (valid, C = O: c = 0 and b solved from a),
    a_identity / b_identity (A = O / B = O, rejected), input_r_minus_1 (valid, x_0 = r - 1)."""
    R = E.R
    m = len(ic) - 1
    x = [synth.scalar("edge-x-%s" % kind, j, seed) for j in range(m)]
    a, b = synth.scalar("edge-a-" + kind, 0, seed), synth.scalar("edge-b-" + kind, 0, seed)
    if kind == "p_identity":
        rest = (ic[0] + sum(xj * icj for xj, icj in zip(x[1:], ic[2:]))) % R
        x[0] = -rest * pow(ic[1], -1, R) % R
    elif kind == "c_identity":
        icx = (ic[0] + sum(xj * icj for xj, icj in zip(x, ic[1:]))) % R
        b = (vk["alpha"] * vk["beta"] + vk["gamma"] * icx) * pow(a, -1, R) % R
        return (a, b, 0), x
    elif kind == "input_r_minus_1":
        if m:
            x[0] = R - 1
    elif kind == "a_identity":
        return (0, b, _groth16_c(vk, ic, a, b, x)), x
    elif kind == "b_identity":
        return (a, 0, _groth16_c(vk, ic, a, b, x)), x
    else:
        raise ValueError(kind)
    return (a, b, _groth16_c(vk, ic, a, b, x)), x


def groth16_mixed_scalars(num_inputs, seed=0):
    """About forty proofs (exponents) with every tamper and edge class the input count allows, plus valid ones:
    -> (vk, ic, proofs, inputs, kinds)."""
    sc, base, base_x = synth.groth16_instance_scalars(28, max(num_inputs, 1), seed)
    vk, ic = sc["vk"], sc["ic"][: num_inputs + 1]
    inputs = [list(x[:num_inputs]) for x in base_x]
    proofs = [(a, b, _groth16_c(vk, ic, a, b, x)) for (a, b, _), x in zip(base, inputs)]
    kinds = ["valid"] * len(proofs)
    pos = 1
    for kind in GROTH16_TAMPER:
        if kind == "input_changed" and not num_inputs:
            continue
        j = pos + 1 if kind == "b_swapped" else None
        groth16_tamper(vk, ic, proofs, inputs, kind, pos, j)
        kinds[pos] = kind
        if j is not None:
            kinds[j] = kind
        pos += 3
    for e, kind in enumerate(GROTH16_EDGE * 2):
        if kind == "p_identity" and not num_inputs:
            continue
        p, x = groth16_edge(vk, ic, kind, seed * 7 + e)
        proofs.append(p)
        inputs.append(x)
        kinds.append(kind)
    return vk, ic, proofs, inputs, kinds


def groth16_points(vk, ic, proofs):
    """Exponents -> (vk dict of points as groth16_instance returns it, [(A, B, C)]); exponent 0 is the identity."""
    vkp = {
        "alpha_g1": E.g1_mul(E.G1_GEN, vk["alpha"]), "beta_g2": E.g2_mul(E.G2_GEN, vk["beta"]),
        "gamma_g2": E.g2_mul(E.G2_GEN, vk["gamma"]), "delta_g2": E.g2_mul(E.G2_GEN, vk["delta"]),
        "gamma_abc_g1": [E.g1_mul(E.G1_GEN, s) for s in ic],
    }
    return vkp, [(E.g1_mul(E.G1_GEN, a), E.g2_mul(E.G2_GEN, b), E.g1_mul(E.G1_GEN, c)) for a, b, c in proofs]
