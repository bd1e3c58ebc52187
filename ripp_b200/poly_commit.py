"""The polynomial-commitment application (ip_proofs/src/applications/poly_commit/mod.rs: KZG :52-131,
BivariatePolynomialCommitment :153-284, UnivariatePolynomialCommitment :286-377; transparent.rs) over the C ABI's
`ripp_pc_*` entry points (csrc/poly_commit.cuh).

Commit is one segmented MSM of the Y polynomials over the shared first-tier bases plus the AFGHO pairing product; open
keeps the powers of x, the row combination y_eval, y_eval_comm, the KZG quotient and the inner-product arguments on the
device; verify is `ripp_pc_verify`, and `verify_batch` checks many openings in one call (`ripp_pc_verify_batch`), one
status per opening: the `AGG_*` constants of `ripp_b200.ip_proofs` (AGG_OK where `verify` accepts, AGG_REJECTED where
it returns False, AGG_MALFORMED / AGG_NOT_IN_SUBGROUP where it raises on the proof's bytes).  Polynomials are coefficient lists of ints (lowest degree first); a bivariate
polynomial is the list of its Y polynomials.  The `*_dev` methods take the coefficients already on the device, row-major
with row length y_degree + 1 (include/ripp_b200.h "Coefficient layout"; a univariate polynomial is already in it), so
that large polynomials skip the host encoding.  Setup takes alpha, beta explicitly (SURVEY.md §8d).  No CPU fallback:
the context fails without a GPU."""
import math

from . import _lib, codec
from .inner_products import default_context
from .ip_proofs import AGG_MALFORMED, AGG_NOT_IN_SUBGROUP, AGG_OK, AGG_REJECTED, vsrs_enc  # noqa: F401 (re-exported)

R = codec.R


def _powers(s, n):
    out, cur = [], 1
    for _ in range(n):
        out.append(cur)
        cur = cur * s % R
    return out


def _gen(ctx, group, exps):
    """exps[i] * generator on the GPU -> DeviceBuffer of affine points."""
    sc = ctx.to_device(codec.fr_vec_enc(exps))
    out = ctx.alloc(len(exps) * (96 if group == 1 else 192))
    (ctx.g1_scale_dev if group == 1 else ctx.g2_scale_dev)(None, sc, len(exps), out)
    ctx.sync()
    sc.free()
    return out


def _v_srs(ctx, alpha, beta):
    g1 = _gen(ctx, 1, [1, beta]).download((2, 24))
    g2 = _gen(ctx, 2, [1, alpha]).download((2, 48))
    return {"g": codec.g1_dec(g1[0]), "h": codec.g2_dec(g2[0]), "g_beta": codec.g1_dec(g1[1]), "h_alpha": codec.g2_dec(g2[1])}


def _upload_fr(ctx, vals):
    """-> (DeviceBuffer or None, length) of Montgomery Fr."""
    vals = list(vals)
    return (ctx.to_device(codec.fr_vec_enc(vals)) if vals else None), len(vals)


def _flat(y_polynomials, m):
    """Y polynomials -> the row-major coefficient list of row length m (rows past the given ones are implicit zeros)."""
    flat = []
    for yp in y_polynomials:
        assert len(yp) <= m  # KZG::commit / Pedersen over m bases (mod.rs:85)
        flat += list(yp) + [0] * (m - len(yp))
    return flat


def _commit_batch_dev(ctx, first, second, coeffs_devs, lengths):
    """ripp_pc_commit_batch_dev under the key (first, second) = ((DeviceBuffer, m), (DeviceBuffer, n))."""
    ctx = ctx or default_context()
    (f, m), (s, n) = first, second
    y_coms = ctx.alloc(max(len(coeffs_devs), 1) * n * 96)
    coms = ctx.pc_commit_batch_dev(f, m, s, n, coeffs_devs, lengths, y_coms)
    return [codec.gt_dec(c) for c in coms], y_coms


def _open_batch_dev(ctx, kind, first, second, srs_g2, coeffs_devs, lengths, y_coms_dev, points):
    ctx = ctx or default_context()
    (f, m), (s, n) = first, second
    xs = [codec.fr_enc(x % R) for x, _ in points]
    ys = [codec.fr_enc(y % R) for _, y in points]
    proofs, ev = ctx.pc_open_batch_dev(kind, f, m, s, n, srs_g2, coeffs_devs, lengths, y_coms_dev, xs, ys)
    return proofs, [codec.fr_dec(e) for e in ev]


def _commit_batch(cls, key, flats, n, ctx):
    """flats[k]: row-major coefficients of polynomial k.  -> list of (com, y_polynomial_coms)."""
    ctx = ctx or default_context()
    bufs = [_upload_fr(ctx, c) for c in flats]
    coms, y_coms = cls.commit_batch_dev(key, [b for b, _ in bufs], [k for _, k in bufs], ctx)
    ys = y_coms.download((max(len(flats), 1) * n, 24))
    return [(com, codec.g1_vec_dec(ys[k * n:(k + 1) * n])) for k, com in enumerate(coms)]


def _open_batch(cls, key, flats, y_polynomial_comms, points, ctx):
    ctx = ctx or default_context()
    bufs = [_upload_fr(ctx, c) for c in flats]
    y_coms = ctx.to_device(codec.g1_vec_enc([p for coms in y_polynomial_comms for p in coms])) if flats else None
    return cls.open_batch_dev(key, [b for b, _ in bufs], [k for _, k in bufs], y_coms, points, ctx)[0]


def _verify_batch(ctx, kind, vsrs, first, second, coms, points, evaluations, proofs):
    """ripp_pc_verify_batch; first / second: (DeviceBuffer, length) or (None, 0).  -> np.uint8 statuses."""
    ctx = ctx or default_context()
    (f, m), (s, n) = first, second
    return ctx.pc_verify_batch(kind, vsrs, f, m, s, n, [codec.gt_enc(c) for c in coms], [codec.fr_enc(x % R) for x, _ in points],
                               [codec.fr_enc(y % R) for _, y in points], [codec.fr_enc(e % R) for e in evaluations], proofs)


def quotient_by_linear(coeffs, z):
    """mod.rs:98-104: polynomial / (X - z), remainder dropped."""
    if len(coeffs) < 2:
        return []
    q, carry = [0] * (len(coeffs) - 1), 0
    for i in range(len(coeffs) - 1, 0, -1):
        carry = (coeffs[i] + z * carry) % R
        q[i - 1] = carry
    return q


class KZG:
    """mod.rs:52-131.  `powers` is a (DeviceBuffer, count) pair of G1 affine points g^(alpha^i)."""

    @staticmethod
    def setup(degree, alpha, beta, ctx=None):
        ctx = ctx or default_context()
        return (_gen(ctx, 1, _powers(alpha, degree + 1)), degree + 1), _v_srs(ctx, alpha, beta)

    @staticmethod
    def commit(powers, coeffs, ctx=None):
        ctx = ctx or default_context()
        c, n = _upload_fr(ctx, coeffs)
        out = ctx.alloc(96)
        ctx.pc_kzg_commit_dev(powers[0], powers[1], c, n, out)
        return codec.g1_dec(out.download(24))

    @staticmethod
    def open(powers, coeffs, point, ctx=None):
        """-> the proof (mod.rs:92-106): the quotient by (X - point) on the device, then one MSM."""
        ctx = ctx or default_context()
        c, n = _upload_fr(ctx, coeffs)
        out = ctx.alloc(96)
        ctx.pc_kzg_open_dev(powers[0], powers[1], c, n, codec.fr_enc(point % R), out)
        return codec.g1_dec(out.download(24))

    @staticmethod
    def verify(v_srs, com, point, evaluation, proof, ctx=None):
        """mod.rs:120-130: e(com - g eval, h) == e(proof, h_alpha - h point), as ONE two-pair product equal to 1."""
        ctx = ctx or default_context()
        return ctx.pc_kzg_verify(vsrs_enc(v_srs), codec.g1_enc(com), codec.fr_enc(point % R), codec.fr_enc(evaluation % R),
                                 codec.g1_enc(proof))


class BivariatePolynomialCommitment:
    """mod.rs:153-284.  srs = dict(h_beta_powers=(DeviceBuffer, 2 x_degree + 1), ck=(DeviceBuffer, x_degree + 1),
    kzg=(DeviceBuffer, y_degree + 1), v_srs=dict)."""

    @staticmethod
    def setup(x_degree, y_degree, alpha, beta, ctx=None):
        ctx = ctx or default_context()
        m = 2 * x_degree + 1
        pb = _powers(beta, m)
        return {
            "h_beta_powers": (_gen(ctx, 2, pb), m),
            "ck": (_gen(ctx, 2, pb[::2]), x_degree + 1),  # SRS::get_commitment_keys: even powers (tipa/mod.rs:114-118)
            "kzg": (_gen(ctx, 1, _powers(alpha, y_degree + 1)), y_degree + 1),
            "v_srs": _v_srs(ctx, alpha, beta),
        }

    @staticmethod
    def commit_dev(srs, coeffs_dev, length, ctx=None):
        """Coefficients on the device (row-major, row length y_degree + 1).  -> (com: GT, y_polynomial_comms: DeviceBuffer
        of x_degree + 1 G1 affine points)."""
        ctx = ctx or default_context()
        n, m = srs["ck"][1], srs["kzg"][1]
        y_coms = ctx.alloc(n * 96)
        com = ctx.pc_commit_dev(srs["kzg"][0], m, srs["ck"][0], n, coeffs_dev, length, y_coms)
        return codec.gt_dec(com), y_coms

    @classmethod
    def commit(cls, srs, y_polynomials, ctx=None):
        """-> (com: GT, y_polynomial_coms: list of G1)."""
        ctx = ctx or default_context()
        assert srs["ck"][1] >= len(y_polynomials)  # mod.rs:186
        c, n = _upload_fr(ctx, _flat(y_polynomials, srs["kzg"][1]))
        com, y_coms = cls.commit_dev(srs, c, n, ctx)
        return com, codec.g1_vec_dec(y_coms.download((srs["ck"][1], 24)))

    @staticmethod
    def open_dev(srs, coeffs_dev, length, y_coms_dev, point, ctx=None):
        """-> (OpeningProof bytes: TIPAWithSSMProof || y_eval_comm || kzg_proof (mod.rs:145-149), evaluation)."""
        ctx = ctx or default_context()
        x, y = point
        n, m = srs["ck"][1], srs["kzg"][1]
        proof, ev = ctx.pc_open_dev(_lib.PC_TRUSTED, srs["kzg"][0], m, srs["ck"][0], n, srs["h_beta_powers"][0], coeffs_dev,
                                    length, y_coms_dev, codec.fr_enc(x % R), codec.fr_enc(y % R))
        return proof, codec.fr_dec(ev)

    @classmethod
    def open(cls, srs, y_polynomials, y_polynomial_comms, point, ctx=None):
        """-> OpeningProof bytes: TIPAWithSSMProof || y_eval_comm || kzg_proof (field order of mod.rs:145-149)."""
        ctx = ctx or default_context()
        assert srs["ck"][1] >= len(y_polynomials)  # mod.rs:211
        c, n = _upload_fr(ctx, _flat(y_polynomials, srs["kzg"][1]))
        y_coms = ctx.to_device(codec.g1_vec_enc(y_polynomial_comms))
        return cls.open_dev(srs, c, n, y_coms, point, ctx)[0]

    @staticmethod
    def commit_batch_dev(srs, coeffs_devs, lengths, ctx=None):
        """Many polynomials under srs in one call.  -> (list of com: GT, y_coms: DeviceBuffer of count x (x_degree + 1) G1,
        polynomial k at element k (x_degree + 1))."""
        return _commit_batch_dev(ctx, srs["kzg"], srs["ck"], coeffs_devs, lengths)

    @staticmethod
    def open_batch_dev(srs, coeffs_devs, lengths, y_coms_dev, points, ctx=None):
        """points[k] = (x, y).  -> (list of OpeningProof bytes, list of evaluations); entry k as open_dev returns it."""
        return _open_batch_dev(ctx, _lib.PC_TRUSTED, srs["kzg"], srs["ck"], srs["h_beta_powers"][0], coeffs_devs, lengths,
                               y_coms_dev, points)

    @classmethod
    def commit_batch(cls, srs, polynomials, ctx=None):
        """polynomials[k]: a list of Y polynomials.  -> list of (com, y_polynomial_coms)."""
        return _commit_batch(cls, srs, [_flat(p, srs["kzg"][1]) for p in polynomials], srs["ck"][1], ctx)

    @classmethod
    def open_batch(cls, srs, polynomials, y_polynomial_comms, points, ctx=None):
        """-> list of OpeningProof bytes."""
        return _open_batch(cls, srs, [_flat(p, srs["kzg"][1]) for p in polynomials], y_polynomial_comms, points, ctx)

    @staticmethod
    def verify(v_srs, com, point, evaluation, proof, ctx=None):
        ctx = ctx or default_context()
        x, y = point
        return ctx.pc_verify(_lib.PC_TRUSTED, vsrs_enc(v_srs), None, 0, None, 0, codec.gt_enc(com), codec.fr_enc(x % R),
                             codec.fr_enc(y % R), codec.fr_enc(evaluation % R), proof)

    @staticmethod
    def verify_batch(v_srs, coms, points, evaluations, proofs, ctx=None):
        """Opening k is (coms[k], points[k] = (x, y), evaluations[k], proofs[k]); openings of different shapes under one
        v_srs may share a call.  -> np.uint8 array of AGG_* statuses, entry k as verify decides opening k alone."""
        return _verify_batch(ctx, _lib.PC_TRUSTED, vsrs_enc(v_srs), (None, 0), (None, 0), coms, points, evaluations, proofs)


class UnivariatePolynomialCommitment:
    """mod.rs:286-377.  The coefficients, read row-major with row length y_degree + 1, are the bivariate form."""

    @staticmethod
    def bivariate_degrees(univariate_degree):
        sqrt = 1 << (math.ceil(math.sqrt(univariate_degree + 1)) - 1).bit_length()  # mod.rs:292-298
        skew = 16 if sqrt >= 32 else sqrt // 2
        return sqrt // skew - 1, sqrt * skew - 1

    @staticmethod
    def degrees_from_srs(srs):
        return (srs["h_beta_powers"][1] - 1) // 2, srs["kzg"][1] - 1

    @staticmethod
    def bivariate_form(degrees, coeffs):
        xd, yd = degrees
        total = (xd + 1) * (yd + 1)
        c = (list(coeffs) + [0] * total)[:total]
        return [c[i * (yd + 1):(i + 1) * (yd + 1)] for i in range(xd + 1)]

    @classmethod
    def setup(cls, degree, alpha, beta, ctx=None):
        xd, yd = cls.bivariate_degrees(degree)
        return BivariatePolynomialCommitment.setup(xd, yd, alpha, beta, ctx)

    @classmethod
    def commit_dev(cls, srs, coeffs_dev, length, ctx=None):
        return BivariatePolynomialCommitment.commit_dev(srs, coeffs_dev, length, ctx)

    @classmethod
    def commit(cls, srs, coeffs, ctx=None):
        ctx = ctx or default_context()
        n, m = srs["ck"][1], srs["kzg"][1]
        c, length = _upload_fr(ctx, list(coeffs)[: n * m])
        com, y_coms = cls.commit_dev(srs, c, length, ctx)
        return com, codec.g1_vec_dec(y_coms.download((n, 24)))

    @classmethod
    def open_dev(cls, srs, coeffs_dev, length, y_coms_dev, point, ctx=None):
        """-> (OpeningProof bytes, evaluation at point)."""
        m = srs["kzg"][1]
        return BivariatePolynomialCommitment.open_dev(srs, coeffs_dev, length, y_coms_dev, (pow(point, m, R), point), ctx)

    @classmethod
    def open(cls, srs, coeffs, y_polynomial_comms, point, ctx=None):
        ctx = ctx or default_context()
        n, m = srs["ck"][1], srs["kzg"][1]
        c, length = _upload_fr(ctx, list(coeffs)[: n * m])
        return cls.open_dev(srs, c, length, ctx.to_device(codec.g1_vec_enc(y_polynomial_comms)), point, ctx)[0]

    @classmethod
    def commit_batch_dev(cls, srs, coeffs_devs, lengths, ctx=None):
        return BivariatePolynomialCommitment.commit_batch_dev(srs, coeffs_devs, lengths, ctx)

    @classmethod
    def open_batch_dev(cls, srs, coeffs_devs, lengths, y_coms_dev, points, ctx=None):
        """points[k] = z_k, opened at (z_k^m, z_k)."""
        m = srs["kzg"][1]
        return BivariatePolynomialCommitment.open_batch_dev(srs, coeffs_devs, lengths, y_coms_dev,
                                                            [(pow(z, m, R), z) for z in points], ctx)

    @classmethod
    def commit_batch(cls, srs, polynomials, ctx=None):
        n, m = srs["ck"][1], srs["kzg"][1]
        return _commit_batch(cls, srs, [list(c)[: n * m] for c in polynomials], n, ctx)

    @classmethod
    def open_batch(cls, srs, polynomials, y_polynomial_comms, points, ctx=None):
        n, m = srs["ck"][1], srs["kzg"][1]
        return _open_batch(cls, srs, [list(c)[: n * m] for c in polynomials], y_polynomial_comms, points, ctx)

    @classmethod
    def verify(cls, v_srs, max_degree, com, point, evaluation, proof, ctx=None):
        _, yd = cls.bivariate_degrees(max_degree)
        return BivariatePolynomialCommitment.verify(v_srs, com, (pow(point, yd + 1, R), point), evaluation, proof, ctx)

    @classmethod
    def verify_batch(cls, v_srs, max_degree, coms, points, evaluations, proofs, ctx=None):
        """points[k] = z_k, checked at (z_k^(y_degree + 1), z_k).  -> np.uint8 AGG_* statuses."""
        _, yd = cls.bivariate_degrees(max_degree)
        return BivariatePolynomialCommitment.verify_batch(v_srs, coms, [(pow(z, yd + 1, R), z) for z in points], evaluations,
                                                          proofs, ctx)


# ------------------------------------------------------------------------------------------------
# Transparent variant (applications/poly_commit/transparent.rs): no trusted setup.  First tier = Pedersen<G1>
# commitments to the Y polynomials (one segmented MSM over the first-tier key), second tier = AFGHO over them.  Openings
# are the two GIPAs with structured scalar message (second tier: MULTIEXP_SSM; first tier: SCALAR_SSM_G1); the
# verifier's final commitment keys are one MSM over each key vector (`ripp_gipa_verify_dev`).
# ck = dict(first=(DeviceBuffer, y_degree + 1) G1 points, second=(DeviceBuffer, x_degree + 1) G2 points).
# ------------------------------------------------------------------------------------------------
class TransparentBivariatePolynomialCommitment:
    """transparent.rs:85-213."""

    @staticmethod
    def setup_from_points(first_tier_ck, second_tier_ck, ctx=None):
        """The reference draws the keys with `random_generators`; here they are given (affine tuples)."""
        ctx = ctx or default_context()
        return {"first": (ctx.to_device(codec.g1_vec_enc(first_tier_ck)), len(first_tier_ck)),
                "second": (ctx.to_device(codec.g2_vec_enc(second_tier_ck)), len(second_tier_ck))}

    @staticmethod
    def commit_dev(ck, coeffs_dev, length, ctx=None):
        """-> (com: GT, y_polynomial_comms: DeviceBuffer of x_degree + 1 G1 affine points)."""
        ctx = ctx or default_context()
        n, m = ck["second"][1], ck["first"][1]
        y_coms = ctx.alloc(n * 96)
        com = ctx.pc_commit_dev(ck["first"][0], m, ck["second"][0], n, coeffs_dev, length, y_coms)
        return codec.gt_dec(com), y_coms

    @classmethod
    def commit(cls, ck, y_polynomials, ctx=None):
        ctx = ctx or default_context()
        assert ck["second"][1] >= len(y_polynomials)  # :106
        c, n = _upload_fr(ctx, _flat(y_polynomials, ck["first"][1]))
        com, y_coms = cls.commit_dev(ck, c, n, ctx)
        return com, codec.g1_vec_dec(y_coms.download((ck["second"][1], 24)))

    @staticmethod
    def open_dev(ck, coeffs_dev, length, y_coms_dev, point, ctx=None):
        """-> (OpeningProof bytes: second_tier_ip_proof || y_eval_comm || first_tier_ip_proof (:79-83), evaluation)."""
        ctx = ctx or default_context()
        x, y = point
        n, m = ck["second"][1], ck["first"][1]
        proof, ev = ctx.pc_open_dev(_lib.PC_TRANSPARENT, ck["first"][0], m, ck["second"][0], n, None, coeffs_dev, length,
                                    y_coms_dev, codec.fr_enc(x % R), codec.fr_enc(y % R))
        return proof, codec.fr_dec(ev)

    @classmethod
    def open(cls, ck, y_polynomials, y_polynomial_comms, point, ctx=None):
        ctx = ctx or default_context()
        assert ck["second"][1] >= len(y_polynomials)  # :137
        c, n = _upload_fr(ctx, _flat(y_polynomials, ck["first"][1]))
        return cls.open_dev(ck, c, n, ctx.to_device(codec.g1_vec_enc(y_polynomial_comms)), point, ctx)[0]

    @staticmethod
    def commit_batch_dev(ck, coeffs_devs, lengths, ctx=None):
        """-> (list of com: GT, y_coms: DeviceBuffer of count x (x_degree + 1) G1)."""
        return _commit_batch_dev(ctx, ck["first"], ck["second"], coeffs_devs, lengths)

    @staticmethod
    def open_batch_dev(ck, coeffs_devs, lengths, y_coms_dev, points, ctx=None):
        """points[k] = (x, y).  -> (list of OpeningProof bytes, list of evaluations)."""
        return _open_batch_dev(ctx, _lib.PC_TRANSPARENT, ck["first"], ck["second"], None, coeffs_devs, lengths, y_coms_dev, points)

    @classmethod
    def commit_batch(cls, ck, polynomials, ctx=None):
        return _commit_batch(cls, ck, [_flat(p, ck["first"][1]) for p in polynomials], ck["second"][1], ctx)

    @classmethod
    def open_batch(cls, ck, polynomials, y_polynomial_comms, points, ctx=None):
        return _open_batch(cls, ck, [_flat(p, ck["first"][1]) for p in polynomials], y_polynomial_comms, points, ctx)

    @staticmethod
    def verify(ck, com, point, evaluation, proof, ctx=None):
        ctx = ctx or default_context()
        x, y = point
        return ctx.pc_verify(_lib.PC_TRANSPARENT, None, ck["first"][0], ck["first"][1], ck["second"][0], ck["second"][1],
                             codec.gt_enc(com), codec.fr_enc(x % R), codec.fr_enc(y % R), codec.fr_enc(evaluation % R), proof)

    @staticmethod
    def verify_batch(ck, coms, points, evaluations, proofs, ctx=None):
        """Opening k is (coms[k], points[k] = (x, y), evaluations[k], proofs[k]) under ck.  -> np.uint8 AGG_* statuses."""
        return _verify_batch(ctx, _lib.PC_TRANSPARENT, None, ck["first"], ck["second"], coms, points, evaluations, proofs)


class TransparentUnivariatePolynomialCommitment:
    """transparent.rs:215-318."""

    @staticmethod
    def bivariate_degrees(univariate_degree):
        sqrt = 1 << (math.ceil(math.sqrt(univariate_degree + 1)) - 1).bit_length()  # :222-227
        skew = 4 if sqrt >= 8 else sqrt // 2
        return sqrt // skew - 1, sqrt * skew - 1

    @staticmethod
    def degrees_from_ck(ck):
        return ck["second"][1] - 1, ck["first"][1] - 1

    @classmethod
    def commit_dev(cls, ck, coeffs_dev, length, ctx=None):
        return TransparentBivariatePolynomialCommitment.commit_dev(ck, coeffs_dev, length, ctx)

    @classmethod
    def commit(cls, ck, coeffs, ctx=None):
        ctx = ctx or default_context()
        n, m = ck["second"][1], ck["first"][1]
        c, length = _upload_fr(ctx, list(coeffs)[: n * m])
        com, y_coms = cls.commit_dev(ck, c, length, ctx)
        return com, codec.g1_vec_dec(y_coms.download((n, 24)))

    @classmethod
    def open_dev(cls, ck, coeffs_dev, length, y_coms_dev, point, ctx=None):
        m = ck["first"][1]
        return TransparentBivariatePolynomialCommitment.open_dev(ck, coeffs_dev, length, y_coms_dev, (pow(point, m, R), point), ctx)

    @classmethod
    def open(cls, ck, coeffs, y_polynomial_comms, point, ctx=None):
        ctx = ctx or default_context()
        n, m = ck["second"][1], ck["first"][1]
        c, length = _upload_fr(ctx, list(coeffs)[: n * m])
        return cls.open_dev(ck, c, length, ctx.to_device(codec.g1_vec_enc(y_polynomial_comms)), point, ctx)[0]

    @classmethod
    def commit_batch_dev(cls, ck, coeffs_devs, lengths, ctx=None):
        return TransparentBivariatePolynomialCommitment.commit_batch_dev(ck, coeffs_devs, lengths, ctx)

    @classmethod
    def open_batch_dev(cls, ck, coeffs_devs, lengths, y_coms_dev, points, ctx=None):
        """points[k] = z_k, opened at (z_k^m, z_k)."""
        m = ck["first"][1]
        return TransparentBivariatePolynomialCommitment.open_batch_dev(ck, coeffs_devs, lengths, y_coms_dev,
                                                                       [(pow(z, m, R), z) for z in points], ctx)

    @classmethod
    def commit_batch(cls, ck, polynomials, ctx=None):
        n, m = ck["second"][1], ck["first"][1]
        return _commit_batch(cls, ck, [list(c)[: n * m] for c in polynomials], n, ctx)

    @classmethod
    def open_batch(cls, ck, polynomials, y_polynomial_comms, points, ctx=None):
        n, m = ck["second"][1], ck["first"][1]
        return _open_batch(cls, ck, [list(c)[: n * m] for c in polynomials], y_polynomial_comms, points, ctx)

    @classmethod
    def verify(cls, ck, com, point, evaluation, proof, ctx=None):
        _, yd = cls.degrees_from_ck(ck)
        return TransparentBivariatePolynomialCommitment.verify(ck, com, (pow(point, yd + 1, R), point), evaluation, proof, ctx)

    @classmethod
    def verify_batch(cls, ck, coms, points, evaluations, proofs, ctx=None):
        """points[k] = z_k, checked at (z_k^(y_degree + 1), z_k).  -> np.uint8 AGG_* statuses."""
        _, yd = cls.degrees_from_ck(ck)
        return TransparentBivariatePolynomialCommitment.verify_batch(ck, coms, [(pow(z, yd + 1, R), z) for z in points],
                                                                     evaluations, proofs, ctx)
