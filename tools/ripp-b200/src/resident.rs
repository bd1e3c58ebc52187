//! Device-resident vectors and the provers / verifiers that keep GIPA's state in HBM across the log n rounds.
//!
//! Replaces (reference paths): `TIPA::setup` (`ip_proofs/src/tipa/mod.rs:150-164`), `TIPA::prove_with_srs_shift`
//! (`:176-231`), `TIPAWithSSM::prove_with_structured_scalar_message` (`tipa/structured_scalar_message.rs:211-268`),
//! `GIPA::prove` (`gipa.rs:108-133`), `aggregate_proofs` / `verify_aggregate_proof`
//! (`applications/groth16_aggregation.rs:77-231`).  Proofs cross the ABI as arkworks' `serialize_uncompressed` bytes
//! and are decoded with the reference's own derived `CanonicalDeserialize`.
use crate::{check, ctx, pack, GIPA_MULTIEXP_SSM, GIPA_PAIRING};
use ark_bls12_381::{Bls12_381, Fr, G1Affine, G1Projective, G2Affine, G2Projective};
use ark_dh_commitments::{
    afgho16::{AFGHOCommitmentG1, AFGHOCommitmentG2},
    identity::IdentityCommitment,
};
use ark_ec::{pairing::PairingOutput, CurveGroup};
use ark_groth16::{Proof, VerifyingKey};
use ark_inner_products::{Error, MultiexponentiationInnerProduct, PairingInnerProduct};
use ark_ip_proofs::tipa::{structured_scalar_message::TIPAWithSSMProof, TIPAProof, VerifierSRS};
use ark_serialize::{CanonicalDeserialize, CanonicalSerialize, Compress};
use blake2::Blake2b;
use ripp_b200_sys as sys;
use std::marker::PhantomData;
use std::os::raw::c_void;

/// Element types that have a packed device layout.
pub trait DeviceElem {
    const BYTES: usize;
}
impl DeviceElem for Fr {
    const BYTES: usize = 32;
}
impl DeviceElem for G1Affine {
    const BYTES: usize = 96;
}
impl DeviceElem for G2Affine {
    const BYTES: usize = 192;
}

/// RAII handle on a device vector (`ripp_dev_alloc` / `ripp_dev_free`).
pub struct DeviceVec<T: DeviceElem> {
    ptr: *mut c_void,
    len: usize,
    _t: PhantomData<T>,
}
unsafe impl<T: DeviceElem> Send for DeviceVec<T> {}

impl<T: DeviceElem> DeviceVec<T> {
    pub fn alloc(len: usize) -> Result<Self, Error> {
        let mut p = std::ptr::null_mut();
        let c = ctx();
        check(unsafe { sys::ripp_dev_alloc(c.raw(), T::BYTES * len.max(1), &mut p) }, len, len)?;
        Ok(DeviceVec { ptr: p, len, _t: PhantomData })
    }
    fn upload_words(words: &[u64], len: usize) -> Result<Self, Error> {
        let v = Self::alloc(len)?;
        if len > 0 {
            let c = ctx();
            check(unsafe { sys::ripp_dev_upload(c.raw(), v.ptr, words.as_ptr() as *const c_void, 8 * words.len()) }, len, len)?;
        }
        Ok(v)
    }
    pub fn download_words(&self) -> Result<Vec<u64>, Error> {
        let mut out = vec![0u64; T::BYTES / 8 * self.len];
        if self.len > 0 {
            let c = ctx();
            check(unsafe { sys::ripp_dev_download(c.raw(), out.as_mut_ptr() as *mut c_void, self.ptr, 8 * out.len()) },
                  self.len, self.len)?;
        }
        Ok(out)
    }
    pub fn len(&self) -> usize {
        self.len
    }
    pub fn is_empty(&self) -> bool {
        self.len == 0
    }
    pub fn ptr(&self) -> *const c_void {
        self.ptr
    }
    pub fn ptr_mut(&self) -> *mut c_void {
        self.ptr
    }
}
impl<T: DeviceElem> Drop for DeviceVec<T> {
    fn drop(&mut self) {
        let c = ctx();
        unsafe { sys::ripp_dev_free(c.raw(), self.ptr) };
    }
}
impl DeviceVec<Fr> {
    pub fn upload_fr(v: &[Fr]) -> Result<Self, Error> {
        Self::upload_words(&pack::pack_fr(v), v.len())
    }
}
impl DeviceVec<G1Affine> {
    pub fn upload_affine(v: &[G1Affine]) -> Result<Self, Error> {
        Self::upload_words(&pack::pack_g1_aff(v), v.len())
    }
    /// `G::normalize_batch` on the host (one shared inversion), then one copy.
    pub fn upload_projective(v: &[G1Projective]) -> Result<Self, Error> {
        Self::upload_affine(&G1Projective::normalize_batch(v))
    }
    pub fn download(&self) -> Result<Vec<G1Affine>, Error> {
        Ok(self.download_words()?.chunks(12).map(pack::get_g1_aff).collect())
    }
}
impl DeviceVec<G2Affine> {
    pub fn upload_affine(v: &[G2Affine]) -> Result<Self, Error> {
        Self::upload_words(&pack::pack_g2_aff(v), v.len())
    }
    pub fn upload_projective(v: &[G2Projective]) -> Result<Self, Error> {
        Self::upload_affine(&G2Projective::normalize_batch(v))
    }
    pub fn download(&self) -> Result<Vec<G2Affine>, Error> {
        Ok(self.download_words()?.chunks(24).map(pack::get_g2_aff).collect())
    }
}

/// The structured reference string of TIPA, resident on the device: g^(alpha^i) and h^(beta^i), i < 2 size - 1.
pub struct GpuSrs {
    pub g_alpha_powers: DeviceVec<G1Affine>,
    pub h_beta_powers: DeviceVec<G2Affine>,
    pub g_beta: G1Affine,
    pub h_alpha: G2Affine,
    pub size: usize,
}

impl GpuSrs {
    /// `TIPA::setup` (`tipa/mod.rs:150-164`).  The two trapdoors are drawn by the caller exactly as the reference does
    /// (`let alpha = Fr::rand(rng); let beta = Fr::rand(rng);`), so a seeded test sees the reference's SRS.
    pub fn setup(alpha: &Fr, beta: &Fr, size: usize) -> Result<Self, Error> {
        let m = 2 * size - 1;
        let g1 = DeviceVec::<G1Affine>::alloc(m)?;
        let g2 = DeviceVec::<G2Affine>::alloc(m)?;
        let (mut gb, mut ha) = ([0u64; 12], [0u64; 24]);
        let c = ctx();
        let st = unsafe {
            sys::ripp_tipa_setup_dev(c.raw(), (alpha.0).0.as_ptr() as *const c_void, (beta.0).0.as_ptr() as *const c_void, size,
                                     g1.ptr_mut(), g2.ptr_mut(), gb.as_mut_ptr() as *mut c_void, ha.as_mut_ptr() as *mut c_void)
        };
        drop(c);
        check(st, size, size)?;
        Ok(GpuSrs { g_alpha_powers: g1, h_beta_powers: g2, g_beta: pack::get_g1_aff(&gb), h_alpha: pack::get_g2_aff(&ha), size })
    }
    /// From an SRS the reference produced (`setup_inner_product`, `groth16_aggregation.rs:68-75`).
    pub fn from_host(srs: &ark_ip_proofs::tipa::SRS<Bls12_381>) -> Result<Self, Error> {
        Ok(GpuSrs {
            g_alpha_powers: DeviceVec::<G1Affine>::upload_projective(&srs.g_alpha_powers)?,
            h_beta_powers: DeviceVec::<G2Affine>::upload_projective(&srs.h_beta_powers)?,
            g_beta: srs.g_beta.into_affine(),
            h_alpha: srs.h_alpha.into_affine(),
            size: (srs.g_alpha_powers.len() + 1) / 2,
        })
    }
    /// `SRS::get_verifier_key` (`tipa/mod.rs:120-127`).
    pub fn verifier_key(&self) -> Result<VerifierSRS<Bls12_381>, Error> {
        use ark_ec::Group;
        Ok(VerifierSRS {
            g: G1Projective::generator(),
            h: G2Projective::generator(),
            g_beta: self.g_beta.into(),
            h_alpha: self.h_alpha.into(),
        })
    }
}

type IpAB = PairingInnerProduct<Bls12_381>;
type IdGT = IdentityCommitment<PairingOutput<Bls12_381>, Fr>;
type IdG1 = IdentityCommitment<G1Projective, Fr>;
pub type ProofAB = TIPAProof<IpAB, AFGHOCommitmentG1<Bls12_381>, AFGHOCommitmentG2<Bls12_381>, IdGT, Bls12_381, Blake2b>;
pub type ProofC =
    TIPAWithSSMProof<MultiexponentiationInnerProduct<G1Projective>, AFGHOCommitmentG1<Bls12_381>, IdG1, Bls12_381, Blake2b>;

fn proof_capacity(n: usize) -> usize {
    let k = usize::BITS as usize - n.leading_zeros() as usize;
    4096 + k * 6 * 600 + 8 * 600
}

/// `TIPA::prove_with_srs_shift` for the pairing instantiation (`PairingInnerProductAB`, `groth16_aggregation.rs:24-31`):
/// message vectors and keys device resident, all log n rounds on the device.
pub fn tipa_prove_ab(srs: &GpuSrs, a: &DeviceVec<G1Affine>, b: &DeviceVec<G2Affine>, ck_a: &DeviceVec<G2Affine>,
                     ck_b: &DeviceVec<G1Affine>, r_shift: &Fr) -> Result<ProofAB, Error> {
    let n = a.len();
    let mut buf = vec![0u8; proof_capacity(n)];
    let mut len = 0usize;
    let c = ctx();
    let st = unsafe {
        sys::ripp_tipa_prove_dev(c.raw(), GIPA_PAIRING, srs.g_alpha_powers.ptr(), srs.h_beta_powers.ptr(), a.ptr(), b.ptr(),
                                 ck_a.ptr(), ck_b.ptr(), n, (r_shift.0).0.as_ptr() as *const c_void, buf.as_mut_ptr(), buf.len(),
                                 &mut len)
    };
    drop(c);
    check(st, n, b.len())?;
    Ok(ProofAB::deserialize_uncompressed_unchecked(&buf[..len])?)
}

/// `TIPAWithSSM::prove_with_structured_scalar_message` for `MultiExpInnerProductC` (`groth16_aggregation.rs:42-48`):
/// `scalars` is the structured vector r^i.
pub fn tipa_prove_c(srs: &GpuSrs, c_vec: &DeviceVec<G1Affine>, scalars: &DeviceVec<Fr>, ck_a: &DeviceVec<G2Affine>)
                    -> Result<ProofC, Error> {
    let n = c_vec.len();
    let mut buf = vec![0u8; proof_capacity(n)];
    let mut len = 0usize;
    let c = ctx();
    let st = unsafe {
        sys::ripp_tipa_prove_dev(c.raw(), GIPA_MULTIEXP_SSM, srs.g_alpha_powers.ptr(), srs.h_beta_powers.ptr(), c_vec.ptr(),
                                 scalars.ptr(), ck_a.ptr(), std::ptr::null(), n, std::ptr::null(), buf.as_mut_ptr(), buf.len(),
                                 &mut len)
    };
    drop(c);
    check(st, n, scalars.len())?;
    Ok(ProofC::deserialize_uncompressed_unchecked(&buf[..len])?)
}

/// The fields of the reference's `AggregateProof` (`groth16_aggregation.rs:58-66`; private there, so the maintainer
/// adds a constructor or the derive).  `bytes` is the exact serialisation, which `verify_aggregate_proof` takes.
pub struct AggregateProofParts {
    pub com_a: PairingOutput<Bls12_381>,
    pub com_b: PairingOutput<Bls12_381>,
    pub com_c: PairingOutput<Bls12_381>,
    pub ip_ab: PairingOutput<Bls12_381>,
    pub agg_c: G1Projective,
    pub tipa_proof_ab: ProofAB,
    pub tipa_proof_c: ProofC,
    pub bytes: Vec<u8>,
}

/// `aggregate_proofs` (`groth16_aggregation.rs:77-160`): the Groth16 proofs stay in host memory as arkworks holds them;
/// one call copies them (1.5 MB for 2^12 proofs) and runs the whole aggregation on the device.
pub fn aggregate_proofs(srs: &GpuSrs, proofs: &[Proof<Bls12_381>]) -> Result<AggregateProofParts, Error> {
    let n = proofs.len();
    let a = pack::pack_g1_aff(&proofs.iter().map(|p| p.a).collect::<Vec<_>>());
    let b = pack::pack_g2_aff(&proofs.iter().map(|p| p.b).collect::<Vec<_>>());
    let cc = pack::pack_g1_aff(&proofs.iter().map(|p| p.c).collect::<Vec<_>>());
    let mut buf = vec![0u8; 8192 + 2 * proof_capacity(n)];
    let mut len = 0usize;
    let c = ctx();
    let st = unsafe {
        sys::ripp_tipp_aggregate(c.raw(), srs.g_alpha_powers.ptr(), srs.h_beta_powers.ptr(), a.as_ptr() as *const c_void,
                                 b.as_ptr() as *const c_void, cc.as_ptr() as *const c_void, n, buf.as_mut_ptr(), buf.len(), &mut len)
    };
    drop(c);
    check(st, n, n)?;
    buf.truncate(len);
    parse_aggregate(buf)
}

/// `aggregate_proofs` from the proofs' bytes, as an aggregation service receives them from untrusted provers: `proofs`
/// holds n ark-groth16 `Proof` records back to back, each written with `serialize_with_mode(compress)` (192 B
/// compressed, 384 B uncompressed), no length prefix.  The library decodes and validates every point on the GPU
/// (flags, canonical coordinates, curve, prime-order subgroup: what `deserialize_with_mode(_, compress, Validate::Yes)`
/// checks) before aggregating; an invalid record fails with a `GpuError` naming the proof, its component and the reason.
pub fn aggregate_proofs_serialized(srs: &GpuSrs, proofs: &[u8], compress: Compress) -> Result<AggregateProofParts, Error> {
    let record = if compress == Compress::Yes { 192 } else { 384 };
    let n = proofs.len() / record;
    let mut buf = vec![0u8; 8192 + 2 * proof_capacity(n)];
    let mut len = 0usize;
    let c = ctx();
    let st = unsafe {
        sys::ripp_tipp_aggregate_serialized(c.raw(), srs.g_alpha_powers.ptr(), srs.h_beta_powers.ptr(), proofs.as_ptr(),
                                            proofs.len(), n, (compress == Compress::Yes) as i32, buf.as_mut_ptr(), buf.len(),
                                            &mut len)
    };
    drop(c);
    check(st, n, n)?;
    buf.truncate(len);
    parse_aggregate(buf)
}

// AggregateProof { com_a, com_b, com_c, ip_ab, agg_c, tipa_proof_ab, tipa_proof_c } (groth16_aggregation.rs:58-66)
fn parse_aggregate(buf: Vec<u8>) -> Result<AggregateProofParts, Error> {
    let mut rd = &buf[..];
    let com_a = PairingOutput::<Bls12_381>::deserialize_uncompressed_unchecked(&mut rd)?;
    let com_b = PairingOutput::<Bls12_381>::deserialize_uncompressed_unchecked(&mut rd)?;
    let com_c = PairingOutput::<Bls12_381>::deserialize_uncompressed_unchecked(&mut rd)?;
    let ip_ab = PairingOutput::<Bls12_381>::deserialize_uncompressed_unchecked(&mut rd)?;
    let agg_c = G1Projective::deserialize_uncompressed_unchecked(&mut rd)?;
    let tipa_proof_ab = ProofAB::deserialize_uncompressed_unchecked(&mut rd)?;
    let tipa_proof_c = ProofC::deserialize_uncompressed_unchecked(&mut rd)?;
    Ok(AggregateProofParts { com_a, com_b, com_c, ip_ab, agg_c, tipa_proof_ab, tipa_proof_c, bytes: buf })
}

/// `verify_aggregate_proof` (`groth16_aggregation.rs:162-231`).  The statement and the proof cross as bytes; the
/// library re-validates every decoded point (curve and prime-order subgroup) and every GT element before use.
pub fn verify_aggregate_proof(v_srs: &VerifierSRS<Bls12_381>, vk: &VerifyingKey<Bls12_381>, public_inputs: &[Vec<Fr>],
                              proof_bytes: &[u8]) -> Result<bool, Error> {
    let mut vsrs = Vec::with_capacity(72);
    vsrs.extend(pack::pack_g1_aff(&[v_srs.g.into_affine()]));
    vsrs.extend(pack::pack_g2_aff(&[v_srs.h.into_affine()]));
    vsrs.extend(pack::pack_g1_aff(&[v_srs.g_beta.into_affine()]));
    vsrs.extend(pack::pack_g2_aff(&[v_srs.h_alpha.into_affine()]));
    let mut vkw = Vec::new();
    vkw.extend(pack::pack_g1_aff(&[vk.alpha_g1]));
    vkw.extend(pack::pack_g2_aff(&[vk.beta_g2, vk.gamma_g2, vk.delta_g2]));
    vkw.extend(pack::pack_g1_aff(&vk.gamma_abc_g1));
    let m = public_inputs.first().map_or(0, |r| r.len());
    assert_eq!(vk.gamma_abc_g1.len(), m + 1); // groth16_aggregation.rs:214
    let inputs: Vec<u64> = public_inputs.iter().flat_map(|row| pack::pack_fr(row)).collect();
    let mut accept = 0i32;
    let c = ctx();
    let st = unsafe {
        sys::ripp_tipp_verify_aggregate(c.raw(), vsrs.as_ptr() as *const c_void, vkw.as_ptr() as *const c_void, m,
                                        inputs.as_ptr() as *const c_void, public_inputs.len(), proof_bytes.as_ptr(),
                                        proof_bytes.len(), &mut accept)
    };
    drop(c);
    check(st, public_inputs.len(), public_inputs.len())?;
    Ok(accept == 1)
}

/// `GIPA::prove` for the pairing instantiation (`gipa.rs:108-133`): the statement (com_a, com_b, t) is checked on the
/// device before proving; a false statement returns `InnerProductArgumentError::InnerProductInvalid`.
pub fn gipa_prove_checked_ab(a: &DeviceVec<G1Affine>, b: &DeviceVec<G2Affine>, ck_a: &DeviceVec<G2Affine>,
                             ck_b: &DeviceVec<G1Affine>, com: (&PairingOutput<Bls12_381>, &PairingOutput<Bls12_381>,
                                                               &PairingOutput<Bls12_381>)) -> Result<Vec<u8>, Error> {
    let n = a.len();
    let mut stmt = Vec::new();
    com.0.serialize_uncompressed(&mut stmt)?;
    com.1.serialize_uncompressed(&mut stmt)?;
    vec![*com.2].serialize_uncompressed(&mut stmt)?; // IdentityOutput(vec![t]): u64 length 1, then the value
    let mut buf = vec![0u8; proof_capacity(n)];
    let mut len = 0usize;
    let c = ctx();
    let st = unsafe {
        sys::ripp_gipa_prove_checked_dev(c.raw(), GIPA_PAIRING, a.ptr(), b.ptr(), ck_a.ptr(), ck_b.ptr(), n, stmt.as_ptr(),
                                         stmt.len(), buf.as_mut_ptr(), buf.len(), &mut len)
    };
    drop(c);
    check(st, n, b.len())?;
    buf.truncate(len);
    Ok(buf)
}
