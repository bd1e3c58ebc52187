//! The polynomial-commitment application on the GPU (`ip_proofs/src/applications/poly_commit/{mod,transparent}.rs`):
//! `KZG`, `BivariatePolynomialCommitment`, `UnivariatePolynomialCommitment` and the transparent variants over the
//! `ripp_pc_*` entry points.  Keys stay device resident (as `GpuSrs`), polynomials are uploaded once as
//! `DeviceVec<Fr>` in the header's coefficient layout: row-major with row length `y_degree + 1`, zeros past the end.  A
//! univariate polynomial is already in that layout.  Opening proofs cross the ABI as the bytes of `OpeningProof` in
//! field order (the reference derives no serialisation for the struct itself); the evaluation comes back with them.
use crate::resident::DeviceVec;
use crate::{check, ctx, pack};
use ark_bls12_381::{Fr, G1Affine, G2Affine};
use ark_ec::{pairing::PairingOutput, CurveGroup};
use ark_inner_products::Error;
use ark_ip_proofs::tipa::VerifierSRS;
use ripp_b200_sys as sys;
use std::os::raw::c_void;

pub const PC_TRUSTED: i32 = 0;
pub const PC_TRANSPARENT: i32 = 1;

fn fr_ptr(f: &Fr) -> *const c_void {
    (f.0).0.as_ptr() as *const c_void
}

fn pack_vsrs(v: &VerifierSRS<ark_bls12_381::Bls12_381>) -> Vec<u64> {
    let mut w = Vec::with_capacity(72);
    w.extend(pack::pack_g1_aff(&[v.g.into_affine()]));
    w.extend(pack::pack_g2_aff(&[v.h.into_affine()]));
    w.extend(pack::pack_g1_aff(&[v.g_beta.into_affine()]));
    w.extend(pack::pack_g2_aff(&[v.h_alpha.into_affine()]));
    w
}

fn proof_capacity(n: usize, m: usize) -> usize {
    let k = |v: usize| usize::BITS as usize - v.leading_zeros() as usize;
    16 * 600 + (k(n) + k(m)) * 6 * 600
}

/// `KZG` (`mod.rs:52-131`) over powers g^(alpha^i) resident on the device.
pub struct Kzg;
impl Kzg {
    /// `KZG::commit` (`mod.rs:85`).
    pub fn commit(powers: &DeviceVec<G1Affine>, coeffs: &DeviceVec<Fr>) -> Result<G1Affine, Error> {
        let out = DeviceVec::<G1Affine>::alloc(1)?;
        let c = ctx();
        let st = unsafe { sys::ripp_pc_kzg_commit_dev(c.raw(), powers.ptr(), powers.len(), coeffs.ptr(), coeffs.len(), out.ptr_mut()) };
        drop(c);
        check(st, coeffs.len(), powers.len())?;
        Ok(out.download()?[0])
    }
    /// `KZG::open` (`mod.rs:98-104`): the quotient by (X - point) on the device, then one MSM.  -> (proof, f(point))
    pub fn open(powers: &DeviceVec<G1Affine>, coeffs: &DeviceVec<Fr>, point: &Fr) -> Result<(G1Affine, Fr), Error> {
        let out = DeviceVec::<G1Affine>::alloc(1)?;
        let ev = DeviceVec::<Fr>::alloc(1)?;
        let c = ctx();
        let st = unsafe {
            sys::ripp_pc_kzg_open_dev(c.raw(), powers.ptr(), powers.len(), coeffs.ptr(), coeffs.len(), fr_ptr(point), out.ptr_mut(),
                                      ev.ptr_mut())
        };
        drop(c);
        check(st, coeffs.len(), powers.len())?;
        Ok((out.download()?[0], pack::get_fr(&ev.download_words()?)))
    }
    /// `KZG::verify` (`mod.rs:120-130`).
    pub fn verify(v_srs: &VerifierSRS<ark_bls12_381::Bls12_381>, com: &G1Affine, point: &Fr, evaluation: &Fr, proof: &G1Affine)
                  -> Result<bool, Error> {
        let (vs, cw, pw) = (pack_vsrs(v_srs), pack::pack_g1_aff(&[*com]), pack::pack_g1_aff(&[*proof]));
        let mut accept = 0i32;
        let c = ctx();
        let st = unsafe {
            sys::ripp_pc_kzg_verify(c.raw(), vs.as_ptr() as *const c_void, cw.as_ptr() as *const c_void, fr_ptr(point),
                                    fr_ptr(evaluation), pw.as_ptr() as *const c_void, &mut accept)
        };
        drop(c);
        check(st, 1, 1)?;
        Ok(accept == 1)
    }
}

/// The keys of one bivariate commitment scheme, device resident.  Trusted (`BivariatePolynomialCommitment`,
/// `mod.rs:153-284`): `first` = the KZG powers g^(alpha^j) (y_degree + 1), `second` = the even powers h^(beta^(2i))
/// (x_degree + 1), `h_beta_powers` = h^(beta^i), i < 2 x_degree + 1, `v_srs` for the verifier.  Transparent
/// (`transparent.rs:85-213`): `first` / `second` are the Pedersen and AFGHO keys, `h_beta_powers` and `v_srs` are None.
pub struct PcKeys {
    pub first: DeviceVec<G1Affine>,
    pub second: DeviceVec<G2Affine>,
    pub h_beta_powers: Option<DeviceVec<G2Affine>>,
    pub v_srs: Option<VerifierSRS<ark_bls12_381::Bls12_381>>,
}

impl PcKeys {
    fn kind(&self) -> i32 {
        if self.h_beta_powers.is_some() { PC_TRUSTED } else { PC_TRANSPARENT }
    }
    pub fn degrees(&self) -> (usize, usize) {
        (self.second.len() - 1, self.first.len() - 1)
    }

    /// `commit` (`mod.rs:186` / `transparent.rs:106-119`): one segmented MSM of the Y polynomials over the first-tier
    /// bases and the AFGHO product with the second-tier key.  -> (com, y_polynomial_comms on the device)
    pub fn commit(&self, coeffs: &DeviceVec<Fr>) -> Result<(PairingOutput<ark_bls12_381::Bls12_381>, DeviceVec<G1Affine>), Error> {
        let (n, m) = (self.second.len(), self.first.len());
        let y_coms = DeviceVec::<G1Affine>::alloc(n)?;
        let mut gt = [0u64; 72];
        let c = ctx();
        let st = unsafe {
            sys::ripp_pc_commit_dev(c.raw(), self.first.ptr(), m, self.second.ptr(), n, coeffs.ptr(), coeffs.len(),
                                    gt.as_mut_ptr() as *mut c_void, y_coms.ptr_mut())
        };
        drop(c);
        check(st, n, m)?;
        Ok((PairingOutput(pack::get_fq12(&gt)), y_coms))
    }

    /// `open` at (x, y) (trusted: `mod.rs:211` on; transparent: `transparent.rs:137` on).  -> (OpeningProof bytes, f(x, y))
    pub fn open(&self, coeffs: &DeviceVec<Fr>, y_coms: &DeviceVec<G1Affine>, point: (&Fr, &Fr)) -> Result<(Vec<u8>, Fr), Error> {
        let (n, m) = (self.second.len(), self.first.len());
        let mut buf = vec![0u8; proof_capacity(n, m)];
        let mut len = 0usize;
        let mut ev = [0u64; 4];
        let g2 = self.h_beta_powers.as_ref().map_or(std::ptr::null(), |h| h.ptr());
        let c = ctx();
        let st = unsafe {
            sys::ripp_pc_open_dev(c.raw(), self.kind(), self.first.ptr(), m, self.second.ptr(), n, g2, coeffs.ptr(), coeffs.len(),
                                  y_coms.ptr(), fr_ptr(point.0), fr_ptr(point.1), buf.as_mut_ptr(), buf.len(), &mut len,
                                  ev.as_mut_ptr() as *mut c_void)
        };
        drop(c);
        check(st, n, m)?;
        buf.truncate(len);
        Ok((buf, pack::get_fr(&ev)))
    }

    /// `commit` of many polynomials under these keys in one call (`ripp_pc_commit_batch_dev`).  -> (the commitments,
    /// the y_polynomial_comms of polynomial k at elements k (x_degree + 1) .. of one device vector)
    pub fn commit_batch(&self, coeffs: &[&DeviceVec<Fr>])
                        -> Result<(Vec<PairingOutput<ark_bls12_381::Bls12_381>>, DeviceVec<G1Affine>), Error> {
        let (n, m, count) = (self.second.len(), self.first.len(), coeffs.len());
        let y_coms = DeviceVec::<G1Affine>::alloc(count.max(1) * n)?;
        let ptrs: Vec<*const c_void> = coeffs.iter().map(|c| c.ptr()).collect();
        let lens: Vec<usize> = coeffs.iter().map(|c| c.len()).collect();
        let mut gt = vec![0u64; 72 * count.max(1)];
        let c = ctx();
        let st = unsafe {
            sys::ripp_pc_commit_batch_dev(c.raw(), self.first.ptr(), m, self.second.ptr(), n, count, ptrs.as_ptr(), lens.as_ptr(),
                                          gt.as_mut_ptr() as *mut c_void, y_coms.ptr_mut())
        };
        drop(c);
        check(st, n, m)?;
        Ok(((0..count).map(|k| PairingOutput(pack::get_fq12(&gt[72 * k..72 * (k + 1)]))).collect(), y_coms))
    }

    /// `open` of polynomial k at points[k] for every k in one call (`ripp_pc_open_batch_dev`), `y_coms` as
    /// `commit_batch` returns it.  -> (OpeningProof bytes, f_k(x_k, y_k)) per polynomial
    pub fn open_batch(&self, coeffs: &[&DeviceVec<Fr>], y_coms: &DeviceVec<G1Affine>, points: &[(Fr, Fr)])
                      -> Result<Vec<(Vec<u8>, Fr)>, Error> {
        let (n, m, count) = (self.second.len(), self.first.len(), coeffs.len());
        assert_eq!(points.len(), count);
        let ptrs: Vec<*const c_void> = coeffs.iter().map(|c| c.ptr()).collect();
        let lens: Vec<usize> = coeffs.iter().map(|c| c.len()).collect();
        let xs = pack::pack_fr(&points.iter().map(|p| p.0).collect::<Vec<_>>());
        let ys = pack::pack_fr(&points.iter().map(|p| p.1).collect::<Vec<_>>());
        let g2 = self.h_beta_powers.as_ref().map_or(std::ptr::null(), |h| h.ptr());
        let mut buf = vec![0u8; count * proof_capacity(n, m)];
        let mut len = 0usize;
        let mut ev = vec![0u64; 4 * count.max(1)];
        let c = ctx();
        let st = unsafe {
            sys::ripp_pc_open_batch_dev(c.raw(), self.kind(), self.first.ptr(), m, self.second.ptr(), n, g2, count, ptrs.as_ptr(),
                                        lens.as_ptr(), y_coms.ptr(), xs.as_ptr() as *const c_void, ys.as_ptr() as *const c_void,
                                        buf.as_mut_ptr(), buf.len(), &mut len, ev.as_mut_ptr() as *mut c_void)
        };
        drop(c);
        check(st, n, m)?;
        Ok((0..count).map(|k| (buf[k * len..(k + 1) * len].to_vec(), pack::get_fr(&ev[4 * k..4 * k + 4]))).collect())
    }

    /// `verify` of an opening of `com` at (x, y) to `evaluation`.
    pub fn verify(&self, com: &PairingOutput<ark_bls12_381::Bls12_381>, point: (&Fr, &Fr), evaluation: &Fr, proof: &[u8])
                  -> Result<bool, Error> {
        let (n, m) = (self.second.len(), self.first.len());
        let vs = self.v_srs.as_ref().map(pack_vsrs);
        let mut gt = Vec::with_capacity(72);
        pack::put_fq12(&mut gt, &com.0);
        let mut accept = 0i32;
        let c = ctx();
        let st = unsafe {
            sys::ripp_pc_verify(c.raw(), self.kind(), vs.as_ref().map_or(std::ptr::null(), |v| v.as_ptr() as *const c_void),
                                self.first.ptr(), m, self.second.ptr(), n, gt.as_ptr() as *const c_void, fr_ptr(point.0),
                                fr_ptr(point.1), fr_ptr(evaluation), proof.as_ptr(), proof.len(), &mut accept)
        };
        drop(c);
        check(st, n, m)?;
        Ok(accept == 1)
    }

    /// `verify` of many openings in one call (`ripp_pc_verify_batch`): opening k is (coms[k], points[k], evaluations[k],
    /// proofs[k]).  -> one `ripp_agg_status` per opening (0 accepted, 1 malformed, 2 not in the subgroup, 3 rejected),
    /// entry k as `verify` decides opening k alone.
    pub fn verify_batch(&self, coms: &[PairingOutput<ark_bls12_381::Bls12_381>], points: &[(Fr, Fr)], evaluations: &[Fr],
                        proofs: &[&[u8]]) -> Result<Vec<u8>, Error> {
        let (n, m, count) = (self.second.len(), self.first.len(), proofs.len());
        assert!(coms.len() == count && points.len() == count && evaluations.len() == count);
        let vs = self.v_srs.as_ref().map(pack_vsrs);
        let mut gt = Vec::with_capacity(72 * count);
        for com in coms {
            pack::put_fq12(&mut gt, &com.0);
        }
        let xs = pack::pack_fr(&points.iter().map(|p| p.0).collect::<Vec<_>>());
        let ys = pack::pack_fr(&points.iter().map(|p| p.1).collect::<Vec<_>>());
        let evs = pack::pack_fr(evaluations);
        let lens: Vec<usize> = proofs.iter().map(|p| p.len()).collect();
        let bytes: Vec<u8> = proofs.iter().flat_map(|p| p.iter().copied()).collect();
        let mut status = vec![0u8; count];
        let mut accepted = 0usize;
        let c = ctx();
        let st = unsafe {
            sys::ripp_pc_verify_batch(c.raw(), self.kind(), vs.as_ref().map_or(std::ptr::null(), |v| v.as_ptr() as *const c_void),
                                      self.first.ptr(), m, self.second.ptr(), n, count, gt.as_ptr() as *const c_void,
                                      xs.as_ptr() as *const c_void, ys.as_ptr() as *const c_void, evs.as_ptr() as *const c_void,
                                      bytes.as_ptr(), bytes.len(), lens.as_ptr(), status.as_mut_ptr(), &mut accepted)
        };
        drop(c);
        check(st, n, m)?;
        Ok(status)
    }
}

/// `UnivariatePolynomialCommitment` (`mod.rs:286-377`) and its transparent twin: the coefficients are the bivariate
/// form, and the point z maps to (z^(y_degree + 1), z).
pub struct Univariate<'a>(pub &'a PcKeys);
impl<'a> Univariate<'a> {
    /// (x_degree, y_degree) of `mod.rs:292-298` (skew 16) or the transparent variant (skew 4).
    pub fn bivariate_degrees(univariate_degree: usize, transparent: bool) -> (usize, usize) {
        let s = ((univariate_degree + 1) as f64).sqrt().ceil() as usize;
        let sqrt = s.next_power_of_two();
        let skew = if transparent { if sqrt >= 8 { 4 } else { sqrt / 2 } } else if sqrt >= 32 { 16 } else { sqrt / 2 };
        (sqrt / skew - 1, sqrt * skew - 1)
    }
    fn point(&self, z: &Fr) -> Fr {
        use ark_ff::Field;
        z.pow([self.0.first.len() as u64])
    }
    pub fn commit(&self, coeffs: &DeviceVec<Fr>) -> Result<(PairingOutput<ark_bls12_381::Bls12_381>, DeviceVec<G1Affine>), Error> {
        self.0.commit(coeffs)
    }
    pub fn open(&self, coeffs: &DeviceVec<Fr>, y_coms: &DeviceVec<G1Affine>, z: &Fr) -> Result<(Vec<u8>, Fr), Error> {
        self.0.open(coeffs, y_coms, (&self.point(z), z))
    }
    pub fn verify(&self, com: &PairingOutput<ark_bls12_381::Bls12_381>, z: &Fr, evaluation: &Fr, proof: &[u8]) -> Result<bool, Error> {
        self.0.verify(com, (&self.point(z), z), evaluation, proof)
    }
    pub fn commit_batch(&self, coeffs: &[&DeviceVec<Fr>])
                        -> Result<(Vec<PairingOutput<ark_bls12_381::Bls12_381>>, DeviceVec<G1Affine>), Error> {
        self.0.commit_batch(coeffs)
    }
    /// polynomial k opened at zs[k], i.e. at (zs[k]^(y_degree + 1), zs[k])
    pub fn open_batch(&self, coeffs: &[&DeviceVec<Fr>], y_coms: &DeviceVec<G1Affine>, zs: &[Fr]) -> Result<Vec<(Vec<u8>, Fr)>, Error> {
        let points: Vec<(Fr, Fr)> = zs.iter().map(|z| (self.point(z), *z)).collect();
        self.0.open_batch(coeffs, y_coms, &points)
    }
    /// opening k checked at (zs[k]^(y_degree + 1), zs[k]); -> one `ripp_agg_status` per opening
    pub fn verify_batch(&self, coms: &[PairingOutput<ark_bls12_381::Bls12_381>], zs: &[Fr], evaluations: &[Fr], proofs: &[&[u8]])
                        -> Result<Vec<u8>, Error> {
        let points: Vec<(Fr, Fr)> = zs.iter().map(|z| (self.point(z), *z)).collect();
        self.0.verify_batch(coms, &points, evaluations, proofs)
    }
}
