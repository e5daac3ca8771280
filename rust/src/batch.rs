//! Batch entry points of `bbs_plus` on the B200 engine: `PublicKey::verify_batch`, `proof_verify_batch`,
//! `proof_gen_batch`, `SecretKey::sign_batch`, over the C ABI of `include/bbs_b200.h` (libbbs_b200.so, hand-written
//! sm_100a CUDA).  The existing single-item API (`PublicKey::verify` src/verify.rs:18-30, `proof_verify`
//! src/proof_verify.rs:19-34, `SecretKey::sign` src/sign.rs:32-43, generic over `Bn254` / `Bls12_381` with
//! `Bn254Const` / `Bls12381Const` and `HashToG1*`) is untouched; this module is added with `pub mod batch;` in lib.rs.
//!
//! Values cross the boundary in their own `CanonicalSerialize` encodings (compressed points, 32-byte little-endian
//! scalars), so nothing here knows a curve's byte layout.  There is no CPU fallback: without a CUDA device every call
//! returns `BatchError::Cuda`.
//!
//! This file cannot be compiled in the engine's build image (no cargo / rustc there); its `extern "C"` block is checked
//! against the header prototype by prototype by tests/test_rust_binding.py, and the same calls are exercised through
//! the ctypes binding (bbs_sign_b200/api.py) by the parity tests.
#![allow(clippy::too_many_arguments)]

use std::os::raw::{c_char, c_void};

use ark_ec::pairing::Pairing;
use ark_ff::Field;
use ark_serialize::{CanonicalDeserialize, CanonicalSerialize};

use crate::{
    constants::{Bls12381Const, Bn254Const, Constants},
    key_gen::{PublicKey, SecretKey},
    proof_gen::{Proof, ProofGenError},
    sign::{Signature, SignatureError},
    utils::{
        core_utilities::calculate_random_scalars,
        interface_utilities::{create_generators, HashToG1},
        utilities_helper::FromOkm,
    },
};

/// Opaque `bbs_ctx` of include/bbs_b200.h.
#[repr(C)]
pub struct BbsCtx {
    _p: [u8; 0],
}
/// Opaque `bbs_issuer_set` of include/bbs_b200.h.
#[repr(C)]
pub struct BbsIssuerSet {
    _p: [u8; 0],
}

// Every symbol include/bbs_b200.h declares, in the header's order.
extern "C" {
    fn bbs_g1_bytes(curve_id: i32) -> usize;
    fn bbs_g2_bytes(curve_id: i32) -> usize;
    fn bbs_signature_bytes(curve_id: i32) -> usize;
    fn bbs_proof_fixed_bytes(curve_id: i32) -> usize;
    fn bbs_last_error() -> *const c_char;
    fn bbs_build_info() -> *const c_char;
    fn bbs_create_generators(curve_id: i32, device: i32, api_id: *const u8, api_id_len: usize, count: u32, out: *mut u8) -> i32;
    fn bbs_ctx_create(curve_id: i32, device: i32, pk: *const u8, generators: *const u8, n_generators: u32, header: *const u8,
                      header_len: usize, api_id: *const u8, api_id_len: usize, out: *mut *mut BbsCtx) -> i32;
    fn bbs_ctx_create_ex(curve_id: i32, device: i32, flags: u32, pk: *const u8, generators: *const u8, n_generators: u32,
                         header: *const u8, header_len: usize, api_id: *const u8, api_id_len: usize, out: *mut *mut BbsCtx) -> i32;
    fn bbs_ctx_destroy(ctx: *mut BbsCtx);
    fn bbs_ctx_domain(ctx: *mut BbsCtx, out_le32: *mut u8) -> i32;
    fn bbs_msg_to_scalars(ctx: *mut BbsCtx, count: usize, msgs: *const u8, offsets: *const u64, out: *mut u8) -> i32;
    fn bbs_core_verify_batch(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msg_scalars: *const u8, n_msgs: u32, status: *mut u8) -> i32;
    fn bbs_verify_batch(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msgs: *const u8, offsets: *const u64, n_msgs: u32,
                        status: *mut u8) -> i32;
    fn bbs_core_sign_batch(ctx: *mut BbsCtx, sk_le32: *const u8, n: usize, msg_scalars: *const u8, n_msgs: u32, sigs_out: *mut u8,
                           b_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_sign_batch(ctx: *mut BbsCtx, sk_le32: *const u8, n: usize, msgs: *const u8, offsets: *const u64, n_msgs: u32,
                      sigs_out: *mut u8, b_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_core_proof_verify_batch(ctx: *mut BbsCtx, n: usize, proofs_fixed: *const u8, commitments: *const u8, commit_off: *const u64,
                                   disclosed_idx: *const u32, disclosed_scalars: *const u8, dis_off: *const u64, ph: *const u8,
                                   ph_len: usize, status: *mut u8) -> i32;
    fn bbs_proof_verify_batch(ctx: *mut BbsCtx, n: usize, proofs_fixed: *const u8, commitments: *const u8, commit_off: *const u64,
                              disclosed_idx: *const u32, dis_msgs: *const u8, dis_msg_off: *const u64, dis_off: *const u64,
                              ph: *const u8, ph_len: usize, status: *mut u8) -> i32;
    fn bbs_core_proof_gen_batch(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msg_scalars: *const u8, n_msgs: u32,
                                disclosed_idx: *const u32, dis_off: *const u64, random_scalars: *const u8, rand_off: *const u64,
                                commit_off: *const u64, ph: *const u8, ph_len: usize, proofs_fixed_out: *mut u8,
                                commitments_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_proof_gen_batch(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msgs: *const u8, offsets: *const u64, n_msgs: u32,
                           disclosed_idx: *const u32, dis_off: *const u64, random_scalars: *const u8, rand_off: *const u64,
                           commit_off: *const u64, ph: *const u8, ph_len: usize, proofs_fixed_out: *mut u8,
                           commitments_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_core_verify_batch_hdr(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msg_scalars: *const u8, n_msgs: u32, headers: *const u8,
                                 hdr_off: *const u64, status: *mut u8) -> i32;
    fn bbs_verify_batch_hdr(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msgs: *const u8, offsets: *const u64, n_msgs: u32,
                            headers: *const u8, hdr_off: *const u64, status: *mut u8) -> i32;
    fn bbs_core_sign_batch_hdr(ctx: *mut BbsCtx, sk_le32: *const u8, n: usize, msg_scalars: *const u8, n_msgs: u32,
                               headers: *const u8, hdr_off: *const u64, sigs_out: *mut u8, b_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_sign_batch_hdr(ctx: *mut BbsCtx, sk_le32: *const u8, n: usize, msgs: *const u8, offsets: *const u64, n_msgs: u32,
                          headers: *const u8, hdr_off: *const u64, sigs_out: *mut u8, b_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_core_proof_verify_batch_hdr(ctx: *mut BbsCtx, n: usize, proofs_fixed: *const u8, commitments: *const u8,
                                       commit_off: *const u64, disclosed_idx: *const u32, disclosed_scalars: *const u8,
                                       dis_off: *const u64, headers: *const u8, hdr_off: *const u64, phs: *const u8,
                                       ph_off: *const u64, status: *mut u8) -> i32;
    fn bbs_proof_verify_batch_hdr(ctx: *mut BbsCtx, n: usize, proofs_fixed: *const u8, commitments: *const u8, commit_off: *const u64,
                                  disclosed_idx: *const u32, dis_msgs: *const u8, dis_msg_off: *const u64, dis_off: *const u64,
                                  headers: *const u8, hdr_off: *const u64, phs: *const u8, ph_off: *const u64, status: *mut u8) -> i32;
    fn bbs_core_proof_gen_batch_hdr(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msg_scalars: *const u8, n_msgs: u32,
                                    disclosed_idx: *const u32, dis_off: *const u64, random_scalars: *const u8, rand_off: *const u64,
                                    commit_off: *const u64, headers: *const u8, hdr_off: *const u64, phs: *const u8,
                                    ph_off: *const u64, proofs_fixed_out: *mut u8, commitments_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_proof_gen_batch_hdr(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msgs: *const u8, offsets: *const u64, n_msgs: u32,
                               disclosed_idx: *const u32, dis_off: *const u64, random_scalars: *const u8, rand_off: *const u64,
                               commit_off: *const u64, headers: *const u8, hdr_off: *const u64, phs: *const u8, ph_off: *const u64,
                               proofs_fixed_out: *mut u8, commitments_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_issuer_set_create(curve_id: i32, device: i32, n_issuers: usize, pks: *const u8, generators: *const u8,
                             n_generators: u32, header: *const u8, header_len: usize, api_id: *const u8, api_id_len: usize,
                             issuer_status: *mut u8, out: *mut *mut BbsIssuerSet) -> i32;
    fn bbs_issuer_set_destroy(set: *mut BbsIssuerSet);
    fn bbs_issuer_set_memory_bytes(set: *mut BbsIssuerSet, shared_bytes: *mut u64) -> u64;
    fn bbs_verify_batch_multi(set: *mut BbsIssuerSet, n: usize, item_issuer: *const u32, sigs: *const u8, msgs: *const u8,
                              offsets: *const u64, n_msgs: u32, status: *mut u8) -> i32;
    fn bbs_core_verify_batch_multi(set: *mut BbsIssuerSet, n: usize, item_issuer: *const u32, sigs: *const u8,
                                   msg_scalars: *const u8, n_msgs: u32, status: *mut u8) -> i32;
    fn bbs_core_proof_verify_batch_multi(set: *mut BbsIssuerSet, n: usize, item_issuer: *const u32, proofs_fixed: *const u8,
                                         commitments: *const u8, commit_off: *const u64, disclosed_idx: *const u32,
                                         disclosed_scalars: *const u8, dis_off: *const u64, ph: *const u8, ph_len: usize,
                                         status: *mut u8) -> i32;
    fn bbs_proof_verify_batch_multi(set: *mut BbsIssuerSet, n: usize, item_issuer: *const u32, proofs_fixed: *const u8,
                                    commitments: *const u8, commit_off: *const u64, disclosed_idx: *const u32, dis_msgs: *const u8,
                                    dis_msg_off: *const u64, dis_off: *const u64, ph: *const u8, ph_len: usize, status: *mut u8) -> i32;
    fn bbs_rlc_partial_core(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msg_scalars: *const u8, n_msgs: u32, seed: *const u8,
                            index_base: u64, parts_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_rlc_partial(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msgs: *const u8, offsets: *const u64, n_msgs: u32,
                       seed: *const u8, index_base: u64, parts_out: *mut u8, status: *mut u8) -> i32;
    fn bbs_rlc_combine(ctx: *mut BbsCtx, n_parts: usize, parts: *const u8, verdict: *mut u8) -> i32;
    fn bbs_rlc_core_verify_batch(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msg_scalars: *const u8, n_msgs: u32,
                                 seed32_or_null: *const u8, verdict: *mut u8) -> i32;
    fn bbs_rlc_verify_batch(ctx: *mut BbsCtx, n: usize, sigs: *const u8, msgs: *const u8, offsets: *const u64, n_msgs: u32,
                            seed32_or_null: *const u8, verdict: *mut u8) -> i32;
    fn bbs_rlc_core_proof_verify_batch(ctx: *mut BbsCtx, n: usize, proofs_fixed: *const u8, commitments: *const u8,
                                       commit_off: *const u64, disclosed_idx: *const u32, disclosed_scalars: *const u8,
                                       dis_off: *const u64, ph: *const u8, ph_len: usize, seed32_or_null: *const u8,
                                       status: *mut u8, combined: *mut u8) -> i32;
    fn bbs_rlc_proof_verify_batch(ctx: *mut BbsCtx, n: usize, proofs_fixed: *const u8, commitments: *const u8, commit_off: *const u64,
                                  disclosed_idx: *const u32, dis_msgs: *const u8, dis_msg_off: *const u64, dis_off: *const u64,
                                  ph: *const u8, ph_len: usize, seed32_or_null: *const u8, status: *mut u8, combined: *mut u8) -> i32;
    fn bbs_rlc_core_proof_verify_batch_hdr(ctx: *mut BbsCtx, n: usize, proofs_fixed: *const u8, commitments: *const u8,
                                           commit_off: *const u64, disclosed_idx: *const u32, disclosed_scalars: *const u8,
                                           dis_off: *const u64, headers: *const u8, hdr_off: *const u64, phs: *const u8,
                                           ph_off: *const u64, seed32_or_null: *const u8, status: *mut u8, combined: *mut u8) -> i32;
    fn bbs_rlc_proof_verify_batch_hdr(ctx: *mut BbsCtx, n: usize, proofs_fixed: *const u8, commitments: *const u8,
                                      commit_off: *const u64, disclosed_idx: *const u32, dis_msgs: *const u8, dis_msg_off: *const u64,
                                      dis_off: *const u64, headers: *const u8, hdr_off: *const u64, phs: *const u8,
                                      ph_off: *const u64, seed32_or_null: *const u8, status: *mut u8, combined: *mut u8) -> i32;
    fn bbs_msg_to_scalars_dev(ctx: *mut BbsCtx, count: usize, d_msgs: *const u8, d_offsets: *const u64, d_out: *mut u8,
                              stream: *mut c_void) -> i32;
    fn bbs_core_verify_batch_dev(ctx: *mut BbsCtx, n: usize, d_sigs: *const u8, d_msg_scalars: *const u8, n_msgs: u32,
                                 d_status: *mut u8, stream: *mut c_void) -> i32;
    fn bbs_verify_batch_dev(ctx: *mut BbsCtx, n: usize, d_sigs: *const u8, d_msgs: *const u8, d_offsets: *const u64, n_msgs: u32,
                            d_status: *mut u8, stream: *mut c_void) -> i32;
    fn bbs_core_sign_batch_dev(ctx: *mut BbsCtx, sk_le32: *const u8, n: usize, d_msg_scalars: *const u8, n_msgs: u32,
                               d_sigs_out: *mut u8, d_b_out: *mut u8, d_status: *mut u8, stream: *mut c_void) -> i32;
    fn bbs_core_proof_verify_batch_dev(ctx: *mut BbsCtx, n: usize, d_proofs_fixed: *const u8, d_commitments: *const u8,
                                       d_commit_off: *const u64, d_disclosed_idx: *const u32, d_disclosed_scalars: *const u8,
                                       d_dis_off: *const u64, d_ph: *const u8, ph_len: usize, d_status: *mut u8,
                                       stream: *mut c_void) -> i32;
    fn bbs_core_verify_batch_hdr_dev(ctx: *mut BbsCtx, n: usize, d_sigs: *const u8, d_msg_scalars: *const u8, n_msgs: u32,
                                     d_headers: *const u8, d_hdr_off: *const u64, d_status: *mut u8, stream: *mut c_void) -> i32;
    fn bbs_core_proof_verify_batch_hdr_dev(ctx: *mut BbsCtx, n: usize, d_proofs_fixed: *const u8, d_commitments: *const u8,
                                           d_commit_off: *const u64, d_disclosed_idx: *const u32, d_disclosed_scalars: *const u8,
                                           d_dis_off: *const u64, d_headers: *const u8, d_hdr_off: *const u64, d_phs: *const u8,
                                           d_ph_off: *const u64, d_status: *mut u8, stream: *mut c_void) -> i32;
    fn bbs_ctx_launch_count(ctx: *mut BbsCtx) -> u64;
    fn bbs_ctx_memory_bytes(ctx: *mut BbsCtx) -> u64;
    fn bbs_ctx_use_per_thread_pairing(ctx: *mut BbsCtx, on: i32) -> i32;
    fn bbs_ctx_set_rlc_windows(ctx: *mut BbsCtx, windows: u32) -> i32;
    fn bbs_ctx_set_g1_split(ctx: *mut BbsCtx, max_items: usize) -> i32;
    fn bbs_ctx_set_pairing_split(ctx: *mut BbsCtx, max_items: usize) -> i32;
    fn bbs_ctx_set_profiling(ctx: *mut BbsCtx, on: i32) -> i32;
    fn bbs_ctx_kernel_times(ctx: *mut BbsCtx, ms: *mut f32, n: i32) -> i32;
    fn bbs_imad_peak(device: i32, iters: i32, mode: i32, gprod_per_s: *mut f64, ms: *mut f32) -> i32;
    fn bbs_selftest_field(curve_id: i32, device: i32, op: i32, n: usize, a: *const u8, b: *const u8, out: *mut u8) -> i32;
    fn bbs_selftest_g1_mul(curve_id: i32, device: i32, n: usize, points: *const u8, scalars: *const u8, out: *mut u8) -> i32;
    fn bbs_selftest_g1(curve_id: i32, device: i32, op: i32, n: usize, p: *const u8, q: *const u8, scalars: *const u8,
                       out: *mut u8) -> i32;
    fn bbs_selftest_pairing(curve_id: i32, device: i32, n: usize, p_points: *const u8, r_points: *const u8, q_point: *const u8,
                            status: *mut u8) -> i32;
}

// per-item status bytes (include/bbs_b200.h BBS_ST_*)
const ST_REJECT: u8 = 0;
const ST_ACCEPT: u8 = 1;
const ST_ERR_MSG_GEN_LEN: u8 = 2;
const ST_ERR_DISCLOSED_INDEX: u8 = 3;
const ST_ERR_IDX_MSG_LEN: u8 = 4;
const ST_ERR_MALFORMED: u8 = 5;
const ST_ERR_DISCLOSED_LEN: u8 = 6;
const ST_ERR_RANDOM_LEN: u8 = 7;
/// `BBS_CTX_PER_ITEM_HEADER`: the context also serves calls with a header per item (`PublicKey::batch_ctx_per_item_header`).
const BBS_CTX_PER_ITEM_HEADER: u32 = 2;
const BBS_OK: i32 = 0;

/// The reference's curve / constants pairing as the ABI's `curve_id` (include/bbs_b200.h `BBS_CURVE_*`).
pub trait CurveId {
    const ID: i32;
}
impl CurveId for Bls12381Const {
    const ID: i32 = 1; // BBS_CURVE_BLS12_381
}
impl CurveId for Bn254Const {
    const ID: i32 = 2; // BBS_CURVE_BN254
}

/// A whole call failed (nothing was computed).
#[derive(Debug, Clone)]
pub enum BatchError {
    /// BBS_E_ARG: null / oversized arguments, an undecodable or off-subgroup public key or generator.
    Argument(String),
    /// BBS_E_CUDA: no device, out of memory, launch failure.
    Cuda(String),
    /// The items of one call must share the message count (the context is built for one `L`).
    RaggedBatch,
}

/// Per-item outcome that is neither `Ok(true)` nor `Ok(false)`.
#[derive(Debug, Clone)]
pub enum ItemError<R> {
    /// The `Err(..)` the reference's function returns for this item.
    Reference(R),
    /// Status 5: an input the reference refuses at deserialisation (undecodable or off-subgroup point, scalar >= r) or on
    /// which it panics (duplicate disclosed index src/proof_verify.rs:179; sk + e == 0 src/sign.rs:129).
    Malformed,
}

fn last_error() -> String {
    unsafe { std::ffi::CStr::from_ptr(bbs_last_error()).to_string_lossy().into_owned() }
}

fn check(rc: i32) -> Result<(), BatchError> {
    match rc {
        BBS_OK => Ok(()),
        -1 => Err(BatchError::Argument(last_error())),
        _ => Err(BatchError::Cuda(last_error())),
    }
}

fn ser<T: CanonicalSerialize>(v: &T, out: &mut Vec<u8>) {
    v.serialize_compressed(out).expect("serialising into a Vec cannot fail");
}

/// Flat bytes + u64 offsets for a list of message lists (item-major): the layout every byte-message entry point takes.
fn pack(messages: &[&[&[u8]]]) -> (Vec<u8>, Vec<u64>) {
    let (mut flat, mut offs) = (Vec::new(), vec![0u64]);
    for item in messages {
        for m in *item {
            flat.extend_from_slice(m);
            offs.push(flat.len() as u64);
        }
    }
    if flat.is_empty() {
        flat.push(0); // never hand the library a dangling pointer
    }
    (flat, offs)
}

fn uniform_len(messages: &[&[&[u8]]]) -> Result<usize, BatchError> {
    let l = messages.first().map_or(0, |m| m.len());
    if messages.iter().any(|m| m.len() != l) {
        return Err(BatchError::RaggedBatch);
    }
    Ok(l)
}

/// Per (GPU, issuer key, header, L) state: decoded key and generators, `calculate_domain`, window tables, line tables.
/// The reference recomputes generators and the domain on every call (src/verify.rs:35, :73-79); here once.
pub struct BatchCtx {
    raw: *mut BbsCtx,
    curve_id: i32,
    l: usize,
}
// The library serialises nothing itself: one context must not be used from two threads at once (include/bbs_b200.h).
unsafe impl Send for BatchCtx {}
impl Drop for BatchCtx {
    fn drop(&mut self) {
        unsafe { bbs_ctx_destroy(self.raw) }
    }
}

impl BatchCtx {
    pub fn n_messages(&self) -> usize {
        self.l
    }

    /// `calculate_domain` of the context (src/utils/core_utilities.rs:24-63), 32 bytes little-endian.
    pub fn domain_le32(&self) -> Result<[u8; 32], BatchError> {
        let mut out = [0u8; 32];
        check(unsafe { bbs_ctx_domain(self.raw, out.as_mut_ptr()) })?;
        Ok(out)
    }
}

impl<E: Pairing> PublicKey<E> {
    /// Builds the per-issuer state on `device` for batches of signatures / proofs over `l` messages under `header`.
    pub fn batch_ctx<H, C>(&self, header: &[u8], l: usize, device: i32) -> Result<BatchCtx, BatchError>
    where
        H: HashToG1<E>,
        C: for<'a> Constants<'a, E> + CurveId,
    {
        let api_id = [C::CIPHERSUITE_ID, b"H2G_HM2S_"].concat(); // src/verify.rs:31
        let (mut pk, mut gens) = (Vec::new(), Vec::new());
        ser(&self.pk, &mut pk);
        for g in create_generators::<E, H>(l + 1, &api_id) {
            ser(&g, &mut gens);
        }
        let mut raw = std::ptr::null_mut();
        check(unsafe {
            bbs_ctx_create(C::ID, device, pk.as_ptr(), gens.as_ptr(), (l + 1) as u32, header.as_ptr(), header.len(),
                           api_id.as_ptr(), api_id.len(), &mut raw)
        })?;
        Ok(BatchCtx { raw, curve_id: C::ID, l })
    }

    /// A context for batches whose items carry their own header (`verify_batch_per_header`, `SecretKey::sign_batch_per_header`,
    /// `proof_verify_batch_per_item`): one per (key, `l`, device) instead of one per header.  Costs one more window table
    /// (Q1's) than `batch_ctx`.
    pub fn batch_ctx_per_item_header<H, C>(&self, l: usize, device: i32) -> Result<BatchCtx, BatchError>
    where
        H: HashToG1<E>,
        C: for<'a> Constants<'a, E> + CurveId,
    {
        let api_id = [C::CIPHERSUITE_ID, b"H2G_HM2S_"].concat();
        let (mut pk, mut gens) = (Vec::new(), Vec::new());
        ser(&self.pk, &mut pk);
        for g in create_generators::<E, H>(l + 1, &api_id) {
            ser(&g, &mut gens);
        }
        let mut raw = std::ptr::null_mut();
        check(unsafe {
            bbs_ctx_create_ex(C::ID, device, BBS_CTX_PER_ITEM_HEADER, pk.as_ptr(), gens.as_ptr(), (l + 1) as u32, std::ptr::null(), 0,
                              api_id.as_ptr(), api_id.len(), &mut raw)
        })?;
        Ok(BatchCtx { raw, curve_id: C::ID, l })
    }

    /// Batch form of `verify` (src/verify.rs:18-50): `result[i]` is what `self.verify(sigs[i], header, messages[i])` returns.
    /// Builds a context for the call; use `batch_ctx` + `verify_batch_with` to amortise it over many calls.
    pub fn verify_batch<F, H, C>(&self, sigs: &[Signature<E, F>], header: &[u8], messages: &[&[&[u8]]])
        -> Result<Vec<Result<bool, ItemError<SignatureError>>>, BatchError>
    where
        F: Field + FromOkm<48, F>,
        H: HashToG1<E>,
        C: for<'a> Constants<'a, E> + CurveId,
    {
        let l = uniform_len(messages)?;
        let ctx = self.batch_ctx::<H, C>(header, l, 0)?;
        verify_batch_with(&ctx, sigs, messages)
    }
}

/// `verify_batch` on an existing context (one issuer key, header and message count for the whole batch).
pub fn verify_batch_with<E: Pairing, F: Field>(ctx: &BatchCtx, sigs: &[Signature<E, F>], messages: &[&[&[u8]]])
    -> Result<Vec<Result<bool, ItemError<SignatureError>>>, BatchError> {
    assert_eq!(sigs.len(), messages.len(), "one message list per signature");
    let l = uniform_len(messages)?;
    let mut sb = Vec::new();
    for s in sigs {
        ser(s, &mut sb); // comp(a) || LE32(e)   (src/sign.rs:18-22)
    }
    let (flat, offs) = pack(messages);
    let mut st = vec![0u8; sigs.len()];
    check(unsafe { bbs_verify_batch(ctx.raw, sigs.len(), sb.as_ptr(), flat.as_ptr(), offs.as_ptr(), l as u32, st.as_mut_ptr()) })?;
    Ok(st.into_iter().map(signature_status).collect())
}

/// Flat bytes + u64 offsets for one byte string per item (headers, presentation headers).
fn pack_items(items: &[&[u8]]) -> (Vec<u8>, Vec<u64>) {
    let (mut flat, mut offs) = (Vec::new(), vec![0u64]);
    for it in items {
        flat.extend_from_slice(it);
        offs.push(flat.len() as u64);
    }
    if flat.is_empty() {
        flat.push(0);
    }
    (flat, offs)
}

/// `verify_batch_with` where item i has its own header: `result[i]` is what `pk.verify(sigs[i], headers[i], messages[i])`
/// returns.  `ctx` comes from `PublicKey::batch_ctx_per_item_header`.
pub fn verify_batch_per_header<E: Pairing, F: Field>(ctx: &BatchCtx, sigs: &[Signature<E, F>], headers: &[&[u8]],
    messages: &[&[&[u8]]]) -> Result<Vec<Result<bool, ItemError<SignatureError>>>, BatchError> {
    assert!(sigs.len() == messages.len() && headers.len() == sigs.len(), "one header and message list per signature");
    let l = uniform_len(messages)?;
    let mut sb = Vec::new();
    for s in sigs {
        ser(s, &mut sb);
    }
    let (flat, offs) = pack(messages);
    let (hdr, hoff) = pack_items(headers);
    let mut st = vec![0u8; sigs.len()];
    check(unsafe {
        bbs_verify_batch_hdr(ctx.raw, sigs.len(), sb.as_ptr(), flat.as_ptr(), offs.as_ptr(), l as u32, hdr.as_ptr(), hoff.as_ptr(),
                             st.as_mut_ptr())
    })?;
    Ok(st.into_iter().map(signature_status).collect())
}

fn signature_status(s: u8) -> Result<bool, ItemError<SignatureError>> {
    match s {
        ST_ACCEPT => Ok(true),
        ST_REJECT => Ok(false),
        ST_ERR_MSG_GEN_LEN => Err(ItemError::Reference(SignatureError::InvalidMessageAndGeneratorsLength)),
        _ => Err(ItemError::Malformed),
    }
}

fn proof_status(s: u8) -> Result<bool, ItemError<ProofGenError>> {
    use ProofGenError::*;
    match s {
        ST_ACCEPT => Ok(true),
        ST_REJECT => Ok(false),
        ST_ERR_MSG_GEN_LEN => Err(ItemError::Reference(InvalidMessageAndGeneratorsLength)),
        ST_ERR_DISCLOSED_INDEX => Err(ItemError::Reference(InvalidDisclosedIndex)),
        ST_ERR_IDX_MSG_LEN => Err(ItemError::Reference(InvalidIndicesAndMessagesLength)),
        ST_ERR_DISCLOSED_LEN => Err(ItemError::Reference(InvalidDisclosedIndicesLength)),
        ST_ERR_RANDOM_LEN => Err(ItemError::Reference(InvalidRandomScalarsAndUndisclosedIndicesLength)),
        _ => Err(ItemError::Malformed),
    }
}

impl<F: Field + FromOkm<48, F>> SecretKey<F> {
    /// Batch form of `sign` (src/sign.rs:32-60): `result[i]` is what `self.sign(messages[i], header)` returns.
    /// `ctx` must have been built from this key's public key (`sk_to_pk`, src/sign.rs:81).
    pub fn sign_batch<E: Pairing<ScalarField = F>>(&self, ctx: &BatchCtx, messages: &[&[&[u8]]])
        -> Result<Vec<Result<Signature<E, F>, ItemError<SignatureError>>>, BatchError> {
        let n = messages.len();
        let l = uniform_len(messages)?;
        let mut sk = Vec::new();
        ser(&self.sk, &mut sk); // LE32; wiped below
        let (flat, offs) = pack(messages);
        let rec = unsafe { bbs_signature_bytes(ctx.curve_id) };
        let (mut out, mut st) = (vec![0u8; n * rec], vec![0u8; n]);
        let rc = unsafe {
            bbs_sign_batch(ctx.raw, sk.as_ptr(), n, flat.as_ptr(), offs.as_ptr(), l as u32, out.as_mut_ptr(),
                           std::ptr::null_mut(), st.as_mut_ptr())
        };
        for b in sk.iter_mut() {
            unsafe { std::ptr::write_volatile(b, 0) }; // SecretKey is Zeroize + ZeroizeOnDrop (src/key_gen.rs:29)
        }
        check(rc)?;
        Ok((0..n)
            .map(|i| match st[i] {
                ST_ACCEPT => Ok(Signature::deserialize_compressed(&out[i * rec..(i + 1) * rec]).expect("library output")),
                ST_ERR_MSG_GEN_LEN => Err(ItemError::Reference(SignatureError::InvalidMessageAndGeneratorsLength)),
                _ => Err(ItemError::Malformed),
            })
            .collect())
    }

    /// `sign_batch` where item i has its own header: `result[i]` is what `self.sign(messages[i], headers[i])` returns.
    /// `ctx` comes from `PublicKey::batch_ctx_per_item_header` of this key's public key.
    pub fn sign_batch_per_header<E: Pairing<ScalarField = F>>(&self, ctx: &BatchCtx, headers: &[&[u8]], messages: &[&[&[u8]]])
        -> Result<Vec<Result<Signature<E, F>, ItemError<SignatureError>>>, BatchError> {
        let n = messages.len();
        assert_eq!(headers.len(), n, "one header per message list");
        let l = uniform_len(messages)?;
        let mut sk = Vec::new();
        ser(&self.sk, &mut sk);
        let (flat, offs) = pack(messages);
        let (hdr, hoff) = pack_items(headers);
        let rec = unsafe { bbs_signature_bytes(ctx.curve_id) };
        let (mut out, mut st) = (vec![0u8; n * rec], vec![0u8; n]);
        let rc = unsafe {
            bbs_sign_batch_hdr(ctx.raw, sk.as_ptr(), n, flat.as_ptr(), offs.as_ptr(), l as u32, hdr.as_ptr(), hoff.as_ptr(),
                               out.as_mut_ptr(), std::ptr::null_mut(), st.as_mut_ptr())
        };
        for b in sk.iter_mut() {
            unsafe { std::ptr::write_volatile(b, 0) };
        }
        check(rc)?;
        Ok((0..n)
            .map(|i| match st[i] {
                ST_ACCEPT => Ok(Signature::deserialize_compressed(&out[i * rec..(i + 1) * rec]).expect("library output")),
                ST_ERR_MSG_GEN_LEN => Err(ItemError::Reference(SignatureError::InvalidMessageAndGeneratorsLength)),
                _ => Err(ItemError::Malformed),
            })
            .collect())
    }
}

/// The ABI splits ark's serialisation of `Proof` (src/proof_gen.rs:29-39) into the fixed fields
/// comp(a_bar)||comp(b_bar)||comp(d)||LE32(e_cap)||LE32(r1_cap)||LE32(r3_cap)||LE32(challenge) and the LE32 commitments.
fn split_proof<E: Pairing, F: Field>(p: &Proof<E, F>, fixed: &mut Vec<u8>, commits: &mut Vec<u8>) {
    ser(&p.a_bar, fixed);
    ser(&p.b_bar, fixed);
    ser(&p.d, fixed);
    ser(&p.e_cap, fixed);
    ser(&p.r1_cap, fixed);
    ser(&p.r3_cap, fixed);
    ser(&p.challenge.scalar, fixed);
    for c in &p.commitments {
        ser(c, commits);
    }
}

/// ... and back: fixed fields + commitments -> ark's `CanonicalSerialize` layout of `Proof` (u64 LE length before the Vec).
fn join_proof<E: Pairing, F: Field>(fixed: &[u8], commits: &[u8]) -> Proof<E, F> {
    let head = fixed.len() - 32;
    let mut blob = Vec::with_capacity(fixed.len() + commits.len() + 8);
    blob.extend_from_slice(&fixed[..head]);
    blob.extend_from_slice(&((commits.len() / 32) as u64).to_le_bytes());
    blob.extend_from_slice(commits);
    blob.extend_from_slice(&fixed[head..]);
    Proof::deserialize_compressed(&blob[..]).expect("library output")
}

/// Batch form of `proof_verify` (src/proof_verify.rs:19-61) on a context built with `l = commitments + disclosed`.
pub fn proof_verify_batch<E: Pairing, F: Field>(ctx: &BatchCtx, proofs: &[Proof<E, F>], ph: &[u8],
    disclosed_messages: &[&[&[u8]]], disclosed_indexes: &[&[usize]])
    -> Result<Vec<Result<bool, ItemError<ProofGenError>>>, BatchError> {
    proof_verify_on(ProofTarget::Ctx(ctx.raw), proofs, ph, disclosed_messages, disclosed_indexes)
}

/// `proof_verify_batch` with a presentation header per proof and, optionally, a header per proof: `result[i]` is what
/// `proof_verify(pk, proofs[i], headers[i], phs[i], ..)` returns.  `headers = None` means the context's header (any context);
/// per-item headers need a context from `PublicKey::batch_ctx_per_item_header`.
pub fn proof_verify_batch_per_item<E: Pairing, F: Field>(ctx: &BatchCtx, proofs: &[Proof<E, F>], headers: Option<&[&[u8]]>,
    phs: &[&[u8]], disclosed_messages: &[&[&[u8]]], disclosed_indexes: &[&[usize]])
    -> Result<Vec<Result<bool, ItemError<ProofGenError>>>, BatchError> {
    assert!(phs.len() == proofs.len() && headers.map_or(true, |h| h.len() == proofs.len()), "one ph (and header) per proof");
    proof_verify_on(ProofTarget::CtxPerItem(ctx.raw, headers, phs), proofs, &[], disclosed_messages, disclosed_indexes)
}

/// `proof_verify_batch` with the pairing checks of the batch folded into one random linear combination
/// (`bbs_rlc_proof_verify_batch`): the same per-item results, where an accepted proof holds except with probability
/// 2^-128 over a coefficient seed the library draws from the OS after it has the batch.  Fast when every proof's pairing
/// holds; a batch in which some proof fails only its pairing costs about as much as `proof_verify_batch`.
pub fn rlc_proof_verify_batch<E: Pairing, F: Field>(ctx: &BatchCtx, proofs: &[Proof<E, F>], ph: &[u8],
    disclosed_messages: &[&[&[u8]]], disclosed_indexes: &[&[usize]])
    -> Result<Vec<Result<bool, ItemError<ProofGenError>>>, BatchError> {
    proof_verify_on(ProofTarget::RlcCtx(ctx.raw), proofs, ph, disclosed_messages, disclosed_indexes)
}

/// `proof_verify_batch_per_item` by one random linear combination, as `rlc_proof_verify_batch`.
pub fn rlc_proof_verify_batch_per_item<E: Pairing, F: Field>(ctx: &BatchCtx, proofs: &[Proof<E, F>], headers: Option<&[&[u8]]>,
    phs: &[&[u8]], disclosed_messages: &[&[&[u8]]], disclosed_indexes: &[&[usize]])
    -> Result<Vec<Result<bool, ItemError<ProofGenError>>>, BatchError> {
    assert!(phs.len() == proofs.len() && headers.map_or(true, |h| h.len() == proofs.len()), "one ph (and header) per proof");
    proof_verify_on(ProofTarget::RlcCtxPerItem(ctx.raw, headers, phs), proofs, &[], disclosed_messages, disclosed_indexes)
}

/// Where a proof batch is verified: under the one key of a context, under a key per proof of an issuer set, or under the
/// key of a context with a ph (and header) per proof; the Rlc forms check the pairings by one random linear combination.
enum ProofTarget<'a> {
    Ctx(*mut BbsCtx),
    Set(*mut BbsIssuerSet, &'a [u32]),
    CtxPerItem(*mut BbsCtx, Option<&'a [&'a [u8]]>, &'a [&'a [u8]]),
    RlcCtx(*mut BbsCtx),
    RlcCtxPerItem(*mut BbsCtx, Option<&'a [&'a [u8]]>, &'a [&'a [u8]]),
}

fn proof_verify_on<E: Pairing, F: Field>(target: ProofTarget, proofs: &[Proof<E, F>], ph: &[u8],
    disclosed_messages: &[&[&[u8]]], disclosed_indexes: &[&[usize]])
    -> Result<Vec<Result<bool, ItemError<ProofGenError>>>, BatchError> {
    let n = proofs.len();
    assert!(disclosed_messages.len() == n && disclosed_indexes.len() == n, "one message / index list per proof");
    // InvalidIndicesAndMessagesLength (src/proof_verify.rs:144-146) is a property of the two host-side lists; the index
    // range check comes first in the reference (:139-143).  Such items are answered here and left out of the call.
    let host_err: Vec<Option<ProofGenError>> = (0..n)
        .map(|i| {
            if disclosed_messages[i].len() == disclosed_indexes[i].len() {
                return None;
            }
            let l = proofs[i].commitments.len() + disclosed_indexes[i].len();
            Some(if disclosed_indexes[i].iter().any(|&x| x >= l) {
                ProofGenError::InvalidDisclosedIndex
            } else {
                ProofGenError::InvalidIndicesAndMessagesLength
            })
        })
        .collect();
    let keep: Vec<usize> = (0..n).filter(|&i| host_err[i].is_none()).collect();
    let (mut fixed, mut commits) = (Vec::new(), Vec::new());
    let (mut coff, mut doff, mut idx) = (vec![0u64], vec![0u64], Vec::<u32>::new());
    let mut kept_msgs: Vec<&[&[u8]]> = Vec::with_capacity(keep.len());
    for &i in &keep {
        split_proof(&proofs[i], &mut fixed, &mut commits);
        coff.push(coff.last().unwrap() + proofs[i].commitments.len() as u64);
        idx.extend(disclosed_indexes[i].iter().map(|&x| x.min(u32::MAX as usize) as u32));
        doff.push(doff.last().unwrap() + disclosed_indexes[i].len() as u64);
        kept_msgs.push(disclosed_messages[i]);
    }
    let (flat, moffs) = pack(&kept_msgs);
    if commits.is_empty() {
        commits.push(0);
    }
    if idx.is_empty() {
        idx.push(0);
    }
    let mut st = vec![0u8; keep.len()];
    if !keep.is_empty() {
        check(match target {
            ProofTarget::Ctx(raw) => unsafe {
                bbs_proof_verify_batch(raw, keep.len(), fixed.as_ptr(), commits.as_ptr(), coff.as_ptr(), idx.as_ptr(), flat.as_ptr(),
                                       moffs.as_ptr(), doff.as_ptr(), ph.as_ptr(), ph.len(), st.as_mut_ptr())
            },
            ProofTarget::Set(raw, item_issuer) => {
                let iss: Vec<u32> = keep.iter().map(|&i| item_issuer[i]).collect();
                unsafe {
                    bbs_proof_verify_batch_multi(raw, keep.len(), iss.as_ptr(), fixed.as_ptr(), commits.as_ptr(), coff.as_ptr(),
                                                 idx.as_ptr(), flat.as_ptr(), moffs.as_ptr(), doff.as_ptr(), ph.as_ptr(), ph.len(),
                                                 st.as_mut_ptr())
                }
            }
            ProofTarget::CtxPerItem(raw, headers, phs) | ProofTarget::RlcCtxPerItem(raw, headers, phs) => {
                // the items kept for the call, with their own ph / header
                let (p, poff) = pack_items(&keep.iter().map(|&i| phs[i]).collect::<Vec<_>>());
                let hs = headers.map(|h| pack_items(&keep.iter().map(|&i| h[i]).collect::<Vec<_>>()));
                let (hp, hoff) = hs.as_ref().map_or((std::ptr::null(), std::ptr::null()), |(h, o)| (h.as_ptr(), o.as_ptr()));
                if matches!(target, ProofTarget::RlcCtxPerItem(..)) {
                    unsafe {
                        bbs_rlc_proof_verify_batch_hdr(raw, keep.len(), fixed.as_ptr(), commits.as_ptr(), coff.as_ptr(), idx.as_ptr(),
                                                       flat.as_ptr(), moffs.as_ptr(), doff.as_ptr(), hp, hoff, p.as_ptr(), poff.as_ptr(),
                                                       std::ptr::null(), st.as_mut_ptr(), std::ptr::null_mut())
                    }
                } else {
                    unsafe {
                        bbs_proof_verify_batch_hdr(raw, keep.len(), fixed.as_ptr(), commits.as_ptr(), coff.as_ptr(), idx.as_ptr(),
                                                   flat.as_ptr(), moffs.as_ptr(), doff.as_ptr(), hp, hoff, p.as_ptr(), poff.as_ptr(),
                                                   st.as_mut_ptr())
                    }
                }
            }
            ProofTarget::RlcCtx(raw) => unsafe {
                bbs_rlc_proof_verify_batch(raw, keep.len(), fixed.as_ptr(), commits.as_ptr(), coff.as_ptr(), idx.as_ptr(), flat.as_ptr(),
                                           moffs.as_ptr(), doff.as_ptr(), ph.as_ptr(), ph.len(), std::ptr::null(), st.as_mut_ptr(),
                                           std::ptr::null_mut())
            },
        })?;
    }
    let mut out: Vec<Result<bool, ItemError<ProofGenError>>> =
        host_err.into_iter().map(|e| Err(ItemError::Reference(e.unwrap_or(ProofGenError::InvalidIndicesAndMessagesLength)))).collect();
    for (k, &i) in keep.iter().enumerate() {
        out[i] = proof_status(st[k]);
    }
    Ok(out)
}

/// Batch form of `proof_gen` (src/proof_gen.rs:78-113).  The `5 + U` random scalars of every proof are drawn here with the
/// crate's own `calculate_random_scalars` (src/utils/core_utilities.rs:70-81), so the device side is a deterministic
/// function of its inputs; with `mocked_calculate_random_scalars` the IRTF proof fixture comes out byte for byte.
pub fn proof_gen_batch<E: Pairing, F: Field + FromOkm<48, F>>(ctx: &BatchCtx, sigs: &[Signature<E, F>], ph: &[u8],
    messages: &[&[&[u8]]], disclosed_indexes: &[&[usize]])
    -> Result<Vec<Result<Proof<E, F>, ItemError<ProofGenError>>>, BatchError> {
    let n = sigs.len();
    assert!(messages.len() == n && disclosed_indexes.len() == n, "one message / index list per signature");
    let l = uniform_len(messages)?;
    let mut sb = Vec::new();
    for s in sigs {
        ser(s, &mut sb);
    }
    let (flat, offs) = pack(messages);
    let (mut idx, mut doff) = (Vec::<u32>::new(), vec![0u64]);
    let (mut rand, mut roff, mut coff) = (Vec::new(), vec![0u64], vec![0u64]);
    for d in disclosed_indexes {
        idx.extend(d.iter().map(|&x| x.min(u32::MAX as usize) as u32));
        doff.push(doff.last().unwrap() + d.len() as u64);
        // the reference sizes the scalars by the raw list (src/proof_gen.rs:143) and commits to the de-duplicated set (:154-158)
        let undisclosed = l.saturating_sub(d.len());
        for r in calculate_random_scalars::<48, F>(5 + undisclosed) {
            ser(&r, &mut rand);
        }
        roff.push(roff.last().unwrap() + (5 + undisclosed) as u64);
        coff.push(coff.last().unwrap() + undisclosed as u64);
    }
    if idx.is_empty() {
        idx.push(0);
    }
    let pf = unsafe { bbs_proof_fixed_bytes(ctx.curve_id) };
    let total_commit = *coff.last().unwrap() as usize;
    let (mut fixed, mut commits, mut st) = (vec![0u8; n * pf], vec![0u8; total_commit.max(1) * 32], vec![0u8; n]);
    let rc = unsafe {
        bbs_proof_gen_batch(ctx.raw, n, sb.as_ptr(), flat.as_ptr(), offs.as_ptr(), l as u32, idx.as_ptr(), doff.as_ptr(), rand.as_ptr(),
                            roff.as_ptr(), coff.as_ptr(), ph.as_ptr(), ph.len(), fixed.as_mut_ptr(), commits.as_mut_ptr(),
                            st.as_mut_ptr())
    };
    for b in rand.iter_mut() {
        unsafe { std::ptr::write_volatile(b, 0) }; // the blinding scalars are secrets of the prover
    }
    check(rc)?;
    Ok((0..n)
        .map(|i| match st[i] {
            ST_ACCEPT => Ok(join_proof(&fixed[i * pf..(i + 1) * pf], &commits[coff[i] as usize * 32..coff[i + 1] as usize * 32])),
            s => Err(proof_status(s).err().unwrap_or(ItemError::Malformed)),
        })
        .collect())
}

/// Many issuer keys over one generator list / header (`bbs_issuer_set_create`): the key is `&self` of every call in the
/// reference (src/verify.rs:18-30), so a batch may name a different issuer per item.  The generator tables are shared;
/// a key costs ~26 KB on BLS12-381.
pub struct IssuerSet {
    raw: *mut BbsIssuerSet,
    /// per key: `true` = usable, `false` = refused like `PublicKey::deserialize_compressed` would (items naming it come
    /// back `ItemError::Malformed`)
    pub usable: Vec<bool>,
}
unsafe impl Send for IssuerSet {}
impl Drop for IssuerSet {
    fn drop(&mut self) {
        unsafe { bbs_issuer_set_destroy(self.raw) }
    }
}

impl IssuerSet {
    pub fn new<E, H, C>(pks: &[PublicKey<E>], header: &[u8], l: usize, device: i32) -> Result<Self, BatchError>
    where
        E: Pairing,
        H: HashToG1<E>,
        C: for<'a> Constants<'a, E> + CurveId,
    {
        let api_id = [C::CIPHERSUITE_ID, b"H2G_HM2S_"].concat();
        let (mut keys, mut gens) = (Vec::new(), Vec::new());
        for pk in pks {
            ser(&pk.pk, &mut keys);
        }
        for g in create_generators::<E, H>(l + 1, &api_id) {
            ser(&g, &mut gens);
        }
        let mut st = vec![0u8; pks.len()];
        let mut raw = std::ptr::null_mut();
        check(unsafe {
            bbs_issuer_set_create(C::ID, device, pks.len(), keys.as_ptr(), gens.as_ptr(), (l + 1) as u32, header.as_ptr(),
                                  header.len(), api_id.as_ptr(), api_id.len(), st.as_mut_ptr(), &mut raw)
        })?;
        Ok(IssuerSet { raw, usable: st.into_iter().map(|s| s == ST_ACCEPT).collect() })
    }

    /// `result[i]` is what `pks[item_issuer[i]].verify(sigs[i], header, messages[i])` returns.
    pub fn verify_batch<E: Pairing, F: Field>(&self, item_issuer: &[u32], sigs: &[Signature<E, F>], messages: &[&[&[u8]]])
        -> Result<Vec<Result<bool, ItemError<SignatureError>>>, BatchError> {
        assert!(item_issuer.len() == sigs.len() && messages.len() == sigs.len());
        let l = uniform_len(messages)?;
        let mut sb = Vec::new();
        for s in sigs {
            ser(s, &mut sb);
        }
        let (flat, offs) = pack(messages);
        let mut st = vec![0u8; sigs.len()];
        check(unsafe {
            bbs_verify_batch_multi(self.raw, sigs.len(), item_issuer.as_ptr(), sb.as_ptr(), flat.as_ptr(), offs.as_ptr(), l as u32,
                                   st.as_mut_ptr())
        })?;
        Ok(st.into_iter().map(signature_status).collect())
    }

    /// `result[i]` is what `pks[item_issuer[i]].proof_verify(proofs[i], header, ph, disclosed_messages[i],
    /// disclosed_indexes[i])` returns (src/proof_verify.rs:19-34).
    pub fn proof_verify_batch<E: Pairing, F: Field>(&self, item_issuer: &[u32], proofs: &[Proof<E, F>], ph: &[u8],
        disclosed_messages: &[&[&[u8]]], disclosed_indexes: &[&[usize]])
        -> Result<Vec<Result<bool, ItemError<ProofGenError>>>, BatchError> {
        assert!(item_issuer.len() == proofs.len());
        proof_verify_on(ProofTarget::Set(self.raw, item_issuer), proofs, ph, disclosed_messages, disclosed_indexes)
    }

    /// (bytes that grow with the number of issuers, shared bytes)
    pub fn memory_bytes(&self) -> (u64, u64) {
        let mut shared = 0u64;
        let per = unsafe { bbs_issuer_set_memory_bytes(self.raw, &mut shared) };
        (per, shared)
    }
}

/// Optional random-linear-combination mode (not in the reference): ONE verdict for the whole batch, wrong with probability
/// 2^-128.  The coefficient seed is drawn inside the library from the OS CSPRNG after it has received the batch.
/// `Ok(true)`: every signature verifies; `Ok(false)`: at least one does not (use `verify_batch_with` to find it).
pub fn rlc_verify_batch<E: Pairing, F: Field>(ctx: &BatchCtx, sigs: &[Signature<E, F>], messages: &[&[&[u8]]])
    -> Result<Result<bool, ItemError<SignatureError>>, BatchError> {
    let l = uniform_len(messages)?;
    let mut sb = Vec::new();
    for s in sigs {
        ser(s, &mut sb);
    }
    let (flat, offs) = pack(messages);
    let mut verdict = 0u8;
    check(unsafe {
        bbs_rlc_verify_batch(ctx.raw, sigs.len(), sb.as_ptr(), flat.as_ptr(), offs.as_ptr(), l as u32, std::ptr::null(), &mut verdict)
    })?;
    Ok(signature_status(verdict))
}

/// Refuses anything but the CUDA build of the library (the host simulation the engine's tests build from the same
/// sources must never be linked into a product).
pub fn assert_cuda_build() {
    let info = unsafe { std::ffi::CStr::from_ptr(bbs_build_info()) }.to_string_lossy();
    assert!(info.starts_with("cuda"), "libbbs_b200 is not a CUDA build: {info}");
}

// The remaining declarations (scalar-level `core_*` entry points, device-buffer variants, sharded RLC, measurement and
// self-test hooks) are bound for completeness; crate code that wants them wraps them like the functions above.
#[allow(dead_code)]
fn _unused_bindings() {
    let _ = (
        bbs_g1_bytes as usize, bbs_g2_bytes as usize, bbs_ctx_create_ex as usize, bbs_create_generators as usize, bbs_msg_to_scalars as usize,
        bbs_core_verify_batch as usize, bbs_core_sign_batch as usize, bbs_core_proof_verify_batch as usize,
        bbs_core_proof_gen_batch as usize, bbs_rlc_partial_core as usize, bbs_rlc_partial as usize, bbs_rlc_combine as usize,
        bbs_rlc_core_verify_batch as usize, bbs_msg_to_scalars_dev as usize, bbs_core_verify_batch_dev as usize,
        bbs_verify_batch_dev as usize, bbs_core_sign_batch_dev as usize, bbs_core_proof_verify_batch_dev as usize,
        bbs_ctx_launch_count as usize, bbs_ctx_memory_bytes as usize, bbs_core_verify_batch_multi as usize, bbs_core_proof_verify_batch_multi as usize, bbs_ctx_use_per_thread_pairing as usize,
        bbs_ctx_set_rlc_windows as usize, bbs_ctx_set_g1_split as usize, bbs_ctx_set_pairing_split as usize, bbs_ctx_set_profiling as usize, bbs_ctx_kernel_times as usize, bbs_imad_peak as usize,
        bbs_selftest_field as usize, bbs_selftest_g1_mul as usize, bbs_selftest_g1 as usize, bbs_selftest_pairing as usize,
        bbs_core_verify_batch_hdr as usize, bbs_core_sign_batch_hdr as usize, bbs_core_proof_verify_batch_hdr as usize,
        bbs_core_proof_gen_batch_hdr as usize, bbs_proof_gen_batch_hdr as usize, bbs_core_verify_batch_hdr_dev as usize,
        bbs_core_proof_verify_batch_hdr_dev as usize, bbs_rlc_core_proof_verify_batch as usize,
        bbs_rlc_core_proof_verify_batch_hdr as usize,
    );
}
