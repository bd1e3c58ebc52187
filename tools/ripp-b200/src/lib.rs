//! `ripp-b200`: the hot path of arkworks-rs/ripp on a B200, behind the reference's own traits.
//!
//! * [`inner_products`] -- `impl InnerProduct` for the pairing, multi-exponentiation and scalar products
//!   (`inner_products/src/lib.rs:40-166`), host slices in, typed arkworks value out.
//! * [`commitments`] -- `impl DoublyHomomorphicCommitment` for AFGHO16 (G1 / G2 messages) and Pedersen
//!   (`dh_commitments/src/afgho16/mod.rs:20-48`, `pedersen/mod.rs:14-27`).  The reference's own types hard-wire
//!   `PairingInnerProduct::<P>` / `MultiexponentiationInnerProduct::<G>`, so the GPU needs its own (identical) structs.
//! * [`resident`] -- device-resident vectors and the provers / verifiers that keep GIPA's state in HBM across rounds:
//!   `TIPA::prove_with_srs_shift`, `TIPAWithSSM::prove_with_structured_scalar_message`, `aggregate_proofs`,
//!   `verify_aggregate_proof`, `TIPA::setup` for given trapdoors.
//! * [`sipp`] -- `SIPP::prove` / `verify` / `product_of_pairings_with_coeffs` (`sipp/src/lib.rs`; BLS12-381 + Blake2s).
//! * [`sipp377`] -- the same three on the reference's own curve, `SIPP<Bls12_377, Blake2s>` (`sipp/src/lib.rs:228-254`).
//!
//! Every value crosses the C ABI as the Montgomery limbs arkworks already holds (`Fp.0 .0`: little-endian `u64`
//! limbs, R = 2^(64 N) -- the same bytes as the ABI's 32-bit limbs on a little-endian host) or as arkworks' own
//! `serialize_uncompressed` bytes.  There is no CPU fallback: without a GPU every entry point fails loudly.
#![allow(clippy::missing_safety_doc)]

pub mod commitments;
pub mod inner_products;
pub mod pack;
pub mod poly_commit;
pub mod resident;
pub mod sipp;
pub mod sipp377;

use ripp_b200_sys as sys;
use std::ffi::CStr;
use std::sync::{Mutex, MutexGuard, OnceLock};

/// Status codes of `include/ripp_b200.h`.
pub const RIPP_OK: i32 = 0;
pub const RIPP_ERR_LEN_MISMATCH: i32 = -1;
pub const RIPP_ERR_NOT_POW2: i32 = -2;
pub const RIPP_ERR_INNER_PRODUCT: i32 = -5;

/// GIPA instantiations (`ripp_gipa_kind`).
pub const GIPA_PAIRING: i32 = 0;
pub const GIPA_MULTIEXP_PEDERSEN: i32 = 1;
pub const GIPA_MULTIEXP_SSM: i32 = 2;

#[derive(Debug)]
pub struct GpuError {
    pub status: i32,
    pub message: String,
}
impl std::fmt::Display for GpuError {
    fn fmt(&self, f: &mut std::fmt::Formatter<'_>) -> std::fmt::Result {
        write!(f, "ripp_b200 status {}: {}", self.status, self.message)
    }
}
impl std::error::Error for GpuError {}

/// One context per process and GPU.  A context is not re-entrant (INTEGRATION.md §3): calls are serialised here,
/// which matches the reference's contract "any thread may call".
pub struct Ctx(*mut sys::ripp_ctx);
unsafe impl Send for Ctx {}

static CTX: OnceLock<Mutex<Ctx>> = OnceLock::new();

/// The process-wide context on device `RIPP_B200_DEVICE` (default 0).  Panics when no GPU is present.
pub fn ctx() -> MutexGuard<'static, Ctx> {
    CTX.get_or_init(|| {
        let device = std::env::var("RIPP_B200_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
        let mut p = std::ptr::null_mut();
        let st = unsafe { sys::ripp_ctx_create(device, &mut p) };
        assert_eq!(st, RIPP_OK, "ripp_b200: {} (there is no CPU fallback)", last_error());
        Mutex::new(Ctx(p))
    })
    .lock()
    .expect("ripp_b200 context poisoned")
}
impl Ctx {
    pub fn raw(&self) -> *mut sys::ripp_ctx {
        self.0
    }
}

pub fn last_error() -> String {
    unsafe { CStr::from_ptr(sys::ripp_last_error_string()) }.to_string_lossy().into_owned()
}

/// Maps a status to the reference's error types: `MessageLengthInvalid` for the two length errors,
/// `InnerProductInvalid` for a failed statement check; everything else (CUDA failure, bad argument) is a `GpuError`.
pub fn check(status: i32, left: usize, right: usize) -> Result<(), ark_inner_products::Error> {
    use ark_inner_products::InnerProductError;
    use ark_ip_proofs::InnerProductArgumentError;
    match status {
        RIPP_OK => Ok(()),
        RIPP_ERR_LEN_MISMATCH => Err(Box::new(InnerProductError::MessageLengthInvalid(left, right))),
        RIPP_ERR_NOT_POW2 => Err(Box::new(InnerProductArgumentError::MessageLengthInvalid(left, right))),
        RIPP_ERR_INNER_PRODUCT => Err(Box::new(InnerProductArgumentError::InnerProductInvalid)),
        s => Err(Box::new(GpuError { status: s, message: last_error() })),
    }
}
