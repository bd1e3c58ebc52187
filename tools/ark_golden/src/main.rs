//! Dumps golden vectors of the arkworks-rs/ripp reference for the synthetic inputs of SURVEY.md §8d
//! (the inputs tests/test_gpu_protocols.py and tests/test_golden.py use), as one JSON object of hex strings.
//!
//! Input derivation (must match oracle/synth.py and ripp_b200/synth.py):
//!   scalar(tag, i, seed) = Fr::from_le_bytes(first 31 bytes of Blake2b-512("ripp-b200/" || tag || LE64(seed) || LE64(i)))
//!   g1_points(tag, n)[i] = scalar(tag, i) * G1::generator(),  g2_points likewise
//!   SRS: alpha = scalar("srs-alpha", 0), beta = scalar("srs-beta", 0), powers as TIPA::setup computes them.
//! Every value is `serialize_uncompressed` bytes, hex encoded, except the `g*c_*` compressed encodings and the
//! `serde_verdict_*` decoder verdicts (hex of "ok" || the decoded point uncompressed, "flags", "invalid" or "other").
//! Usage: cargo run --release -p ark-golden -- <path of tests/golden/serde_cases.txt> > tests/golden/ark_golden.json
use ark_bls12_381::{Bls12_381, Fr, G1Projective as G1, G2Projective as G2};
use ark_dh_commitments::{
    afgho16::{AFGHOCommitmentG1, AFGHOCommitmentG2},
    identity::{HomomorphicPlaceholderValue, IdentityCommitment},
    pedersen::PedersenCommitment,
    DoublyHomomorphicCommitment,
};
use ark_ec::{pairing::PairingOutput, Group};
use ark_ff::PrimeField;
use ark_inner_products::{
    InnerProduct, MultiexponentiationInnerProduct, PairingInnerProduct, ScalarInnerProduct,
};
use ark_ip_proofs::{
    gipa::GIPA,
    tipa::{
        structured_generators_scalar_power,
        structured_scalar_message::{structured_scalar_power, TIPAWithSSM},
        SRS, TIPA,
    },
};
use ark_serialize::CanonicalSerialize;
use ark_sipp::{product_of_pairings_with_coeffs, SIPP};
use ark_ec::CurveGroup;
use blake2::{Blake2b, Blake2s};
use digest::Digest;

const N: usize = 8;

fn scalar(tag: &str, i: u64) -> Fr {
    let mut h = Blake2b::new();
    h.update(b"ripp-b200/");
    h.update(tag.as_bytes());
    h.update(&0u64.to_le_bytes());
    h.update(&i.to_le_bytes());
    Fr::from_le_bytes_mod_order(&h.finalize()[..31])
}
fn scalars(tag: &str, n: usize) -> Vec<Fr> {
    (0..n as u64).map(|i| scalar(tag, i)).collect()
}
fn g1_points(tag: &str, n: usize) -> Vec<G1> {
    scalars(tag, n).iter().map(|s| G1::generator() * s).collect()
}
fn g2_points(tag: &str, n: usize) -> Vec<G2> {
    scalars(tag, n).iter().map(|s| G2::generator() * s).collect()
}
fn hex<T: CanonicalSerialize>(v: &T) -> String {
    let mut b = Vec::new();
    v.serialize_uncompressed(&mut b).unwrap();
    b.iter().map(|x| format!("{:02x}", x)).collect()
}
fn srs(n: usize) -> SRS<Bls12_381> {
    // tipa/mod.rs:150-164 with alpha, beta fixed instead of drawn from the rng
    let (alpha, beta) = (scalar("srs-alpha", 0), scalar("srs-beta", 0));
    let (g, h) = (G1::generator(), G2::generator());
    SRS {
        g_alpha_powers: structured_generators_scalar_power(2 * n - 1, &g, &alpha),
        h_beta_powers: structured_generators_scalar_power(2 * n - 1, &h, &beta),
        g_beta: g * beta,
        h_alpha: h * alpha,
    }
}

/// `serde_case_<group>_<c|u>_<name> <hex>` lines of tests/golden/serde_cases.txt; its path is the first argument.
fn serde_cases() -> Vec<(String, Vec<u8>)> {
    let path = std::env::args().nth(1).unwrap_or_else(|| "serde_cases.txt".into());
    let text = std::fs::read_to_string(&path).expect("pass the path of tests/golden/serde_cases.txt");
    let unhex = |h: &str| (0..h.len()).step_by(2).map(|i| u8::from_str_radix(&h[i..i + 2], 16).unwrap()).collect::<Vec<u8>>();
    text.lines()
        .filter_map(|l| {
            let mut it = l.split_whitespace();
            Some((it.next()?.to_string(), unhex(it.next()?)))
        })
        .collect()
}

type GC1 = AFGHOCommitmentG1<Bls12_381>;
type GC2 = AFGHOCommitmentG2<Bls12_381>;
type SC1 = PedersenCommitment<G1>;
type PIP = PairingInnerProduct<Bls12_381>;
type MIP = MultiexponentiationInnerProduct<G1>;
type IPCGT = IdentityCommitment<PairingOutput<Bls12_381>, Fr>;
type IPCG1 = IdentityCommitment<G1, Fr>;

fn main() {
    let mut out: Vec<(String, String)> = Vec::new();
    let ck_t = HomomorphicPlaceholderValue;
    out.push(("scalar_gipa-b_0".into(), hex(&scalar("gipa-b", 0))));
    out.push(("g1_gipa-a_0".into(), hex(&g1_points("gipa-a", 1)[0].into_affine())));
    out.push(("g2_gipa-b_0".into(), hex(&g2_points("gipa-b", 1)[0].into_affine())));

    // inner products and commitments (inner_products/src/lib.rs, dh_commitments/src/**)
    let (a, b) = (g1_points("gipa-a", N), g2_points("gipa-b", N));
    let (v, w) = (g2_points("gipa-v", N), g1_points("gipa-w", N));
    let t = PIP::inner_product(&a, &b).unwrap();
    out.push(("pairing_ip_n8".into(), hex(&t)));
    let com_a = GC1::commit(&v, &a).unwrap();
    let com_b = GC2::commit(&w, &b).unwrap();
    out.push(("afgho_g1_commit_n8".into(), hex(&com_a)));
    out.push(("afgho_g2_commit_n8".into(), hex(&com_b)));
    let fb = scalars("gipa-b", N);
    out.push(("msm_g1_n8".into(), hex(&MIP::inner_product(&a, &fb).unwrap().into_affine())));
    out.push(("scalar_ip_n8".into(), hex(&ScalarInnerProduct::<Fr>::inner_product(&scalars("gipa-a", N), &fb).unwrap())));

    // GIPA, pairing instantiation (gipa.rs:470-497)
    type PairingGIPA = GIPA<PIP, GC1, GC2, IPCGT, Blake2b>;
    let com_t = IPCGT::commit(&vec![ck_t.clone()], &vec![t.clone()]).unwrap();
    let proof = PairingGIPA::prove((&a, &b, &t), (&v, &w, &ck_t), (&com_a, &com_b, &com_t)).unwrap();
    out.push(("gipa_pairing_n8_proof".into(), hex(&proof)));

    // GIPA, multiexponentiation instantiation (gipa.rs:499-528)
    type MultiExpGIPA = GIPA<MIP, GC1, SC1, IPCG1, Blake2b>;
    let tm = MIP::inner_product(&a, &fb).unwrap();
    let com_bm = SC1::commit(&w, &fb).unwrap();
    let com_tm = IPCG1::commit(&vec![ck_t.clone()], &vec![tm.clone()]).unwrap();
    let proof = MultiExpGIPA::prove((&a, &fb, &tm), (&v, &w, &ck_t), (&com_a, &com_bm, &com_tm)).unwrap();
    out.push(("gipa_multiexp_n8_proof".into(), hex(&proof)));

    // TIPA, pairing instantiation (tipa/mod.rs:450-476): keys = even SRS powers
    type PairingTIPA = TIPA<PIP, GC1, GC2, IPCGT, Bls12_381, Blake2b>;
    let s = srs(N);
    let (ck_a, ck_b) = s.get_commitment_keys();
    let proof = PairingTIPA::prove(&s, (&a, &b), (&ck_a, &ck_b, &ck_t)).unwrap();
    out.push(("tipa_pairing_n8_proof".into(), hex(&proof)));
    out.push(("tipa_pairing_n8_com_a".into(), hex(&GC1::commit(&ck_a, &a).unwrap())));

    // TIPA with structured scalar message (structured_scalar_message.rs:360-390)
    type SsmTIPA = TIPAWithSSM<MIP, GC1, IPCG1, Bls12_381, Blake2b>;
    let sb = scalar("ssm-b", 0);
    let bvec = structured_scalar_power(N, &sb);
    let a2 = g1_points("ssm-a", N);
    let proof = SsmTIPA::prove_with_structured_scalar_message(&s, (&a2, &bvec), (&ck_a, &ck_t)).unwrap();
    out.push(("tipa_ssm_n8_proof".into(), hex(&proof)));

    // SIPP on BLS12-381 + Blake2s (sipp/src/lib.rs:42-106, 184-217)
    let sa: Vec<_> = g1_points("sipp-a", N).iter().map(|p| p.into_affine()).collect();
    let sbp: Vec<_> = g2_points("sipp-b", N).iter().map(|p| p.into_affine()).collect();
    let sr = scalars("sipp-r", N);
    let z = product_of_pairings_with_coeffs::<Bls12_381>(&sa, &sbp, &sr);
    out.push(("sipp_n8_value".into(), hex(&z)));
    // `Proof::gt_elems` is private and `Proof` has no CanonicalSerialize (sipp/src/lib.rs:32-34): the transcript can
    // only be dumped with a one-word upstream patch (`pub gt_elems`), enabled here by `--features sipp-proof`.
    let proof = SIPP::<Bls12_381, Blake2s>::prove(&sa, &sbp, &sr, z).unwrap();
    assert!(SIPP::<Bls12_381, Blake2s>::verify(&sa, &sbp, &sr, z, &proof).unwrap());
    #[cfg(feature = "sipp-proof")]
    {
        let mut pb = Vec::new();
        for (l, r) in proof.gt_elems.iter() {
            l.serialize_uncompressed(&mut pb).unwrap();
            r.serialize_uncompressed(&mut pb).unwrap();
        }
        out.push(("sipp_n8_proof".into(), pb.iter().map(|x| format!("{:02x}", x)).collect()));
    }

    // SIPP on the reference's OWN curve, BLS12-377 + Blake2s (sipp/src/lib.rs:228-254).  The goldens are self-describing:
    // the two generators are dumped, the inputs are scalar(tag, i) * generator with the same 31-byte scalars.
    {
        use ark_bls12_377::{Bls12_377, Fr as Fr7, G1Projective as G17, G2Projective as G27};
        let sc7 = |tag: &str, n: usize| -> Vec<Fr7> {
            (0..n as u64)
                .map(|i| {
                    let mut h = Blake2b::new();
                    h.update(b"ripp-b200/");
                    h.update(tag.as_bytes());
                    h.update(&0u64.to_le_bytes());
                    h.update(&i.to_le_bytes());
                    Fr7::from_le_bytes_mod_order(&h.finalize()[..31])
                })
                .collect()
        };
        out.push(("bls12_377_g1_generator".into(), hex(&G17::generator().into_affine())));
        out.push(("bls12_377_g2_generator".into(), hex(&G27::generator().into_affine())));
        let a7: Vec<_> = sc7("s377-a", N).iter().map(|s| (G17::generator() * s).into_affine()).collect();
        let b7: Vec<_> = sc7("s377-b", N).iter().map(|s| (G27::generator() * s).into_affine()).collect();
        let r7 = sc7("s377-r", N);
        out.push(("bls12_377_g1_s377-a_0".into(), hex(&a7[0])));
        out.push(("bls12_377_g2_s377-b_0".into(), hex(&b7[0])));
        let z7 = product_of_pairings_with_coeffs::<Bls12_377>(&a7, &b7, &r7);
        out.push(("bls12_377_sipp_n8_value".into(), hex(&z7)));
        let proof7 = SIPP::<Bls12_377, Blake2s>::prove(&a7, &b7, &r7, z7).unwrap();
        assert!(SIPP::<Bls12_377, Blake2s>::verify(&a7, &b7, &r7, z7, &proof7).unwrap());
        #[cfg(feature = "sipp-proof")]
        {
            let mut pb = Vec::new();
            for (l, r) in proof7.gt_elems.iter() {
                l.serialize_uncompressed(&mut pb).unwrap();
                r.serialize_uncompressed(&mut pb).unwrap();
            }
            out.push(("bls12_377_sipp_n8_proof".into(), pb.iter().map(|x| format!("{:02x}", x)).collect()));
        }
    }

    // Point encodings for the validating decoders (oracle/serde.py de_g1 / de_g2, csrc/serde.cuh): compressed forms
    // of the points above, and arkworks' verdict (deserialize_with_mode, Validate::Yes) on every encoding listed in
    // tests/golden/serde_cases.txt (oracle/serde_cases.py named_cases: each flag rule, x = p, an x off the curve, a point
    // off the subgroup, valid points), as `serde_verdict_<group>_<c|u>_<name>`.
    {
        use ark_bls12_381::{G1Affine, G2Affine};
        use ark_serialize::{CanonicalDeserialize, Compress, SerializationError, Validate};
        let comp = |v: &dyn Fn(&mut Vec<u8>)| -> String {
            let mut b = Vec::new();
            v(&mut b);
            b.iter().map(|x| format!("{:02x}", x)).collect()
        };
        let g1 = g1_points("gipa-a", 1)[0].into_affine();
        let g2 = g2_points("gipa-b", 1)[0].into_affine();
        out.push(("g1c_gipa-a_0".into(), comp(&|b| g1.serialize_compressed(b).unwrap())));
        out.push(("g2c_gipa-b_0".into(), comp(&|b| g2.serialize_compressed(b).unwrap())));
        out.push(("g1c_generator".into(), comp(&|b| G1::generator().into_affine().serialize_compressed(b).unwrap())));
        out.push(("g2c_generator".into(), comp(&|b| G2::generator().into_affine().serialize_compressed(b).unwrap())));
        // verdicts: "ok:<uncompressed bytes of the point>" or the SerializationError variant
        let verdict = |r: Result<Vec<u8>, SerializationError>| -> String {
            match r {
                Ok(b) => format!("6f6b{}", b.iter().map(|x| format!("{:02x}", x)).collect::<String>()),  // "ok" || point
                Err(SerializationError::UnexpectedFlags) => "666c616773".into(),                          // "flags"
                Err(SerializationError::InvalidData) => "696e76616c6964".into(),                          // "invalid"
                Err(_) => "6f74686572".into(),                                                            // "other"
            }
        };
        let cases: Vec<(String, Vec<u8>)> = serde_cases();
        for (key, bytes) in cases {
            let compressed = key.contains("_c_");
            let mode = if compressed { Compress::Yes } else { Compress::No };
            let r = if key.starts_with("serde_case_1_") {
                G1Affine::deserialize_with_mode(&bytes[..], mode, Validate::Yes).map(|p| {
                    let mut b = Vec::new();
                    p.serialize_uncompressed(&mut b).unwrap();
                    b
                })
            } else {
                G2Affine::deserialize_with_mode(&bytes[..], mode, Validate::Yes).map(|p| {
                    let mut b = Vec::new();
                    p.serialize_uncompressed(&mut b).unwrap();
                    b
                })
            };
            out.push((key.replace("serde_case_", "serde_verdict_"), verdict(r)));
        }
    }

    // AggregateProof has private fields and no CanonicalSerialize (groth16_aggregation.rs:58-66): its parts are
    // covered by the two TIPA goldens above; add `#[derive(CanonicalSerialize)]` upstream to dump it whole.
    println!("{{");
    for (i, (k, v)) in out.iter().enumerate() {
        println!("  \"{}\": \"{}\"{}", k, v, if i + 1 < out.len() { "," } else { "" });
    }
    println!("}}");
}
