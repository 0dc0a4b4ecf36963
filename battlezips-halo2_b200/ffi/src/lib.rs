//! bzhalo2-sys -- Rust side of the drop-in boundary: raw bindings of `include/bzhalo2.h` (sys.rs, generated from the header) and
//! the wrappers the patched `halo2_proofs 0.2.0` calls (`halo2_proofs-0.2.0-bz.patch` next to this crate).
//!
//! UNBUILT SOURCE: there is no cargo / rustc in the build image or on the GPU box (DESIGN.md §0); what CI executes drives the
//! same C symbols through ctypes.  Kept complete and reviewable against the header: `tests/test_abi_exports.py` checks that
//! sys.rs declares every symbol of the header with the header's arity.
//!
//! Layout contract (SURVEY §8b): `pasta_curves::{Fp, Fq}` are `#[repr(transparent)]` wrappers of `[u64; 4]` in Montgomery
//! form = the 32-byte element of the ABI, so `&[Fp]` crosses as a pointer.  Affine points are marshalled explicitly as
//! x || y (`EpAffine`'s struct layout is not `repr(C)`); the identity is 64 zero bytes.
#![allow(non_camel_case_types)]
use std::cell::RefCell;
use std::os::raw::{c_int, c_void};

use ff::{Field, PrimeField};
use group::Curve;
use pasta_curves::arithmetic::{CurveAffine, FieldExt};
use pasta_curves::{vesta, Fp, Fq};
use rand_core::RngCore;

pub mod sys;
pub use sys::*;

#[repr(C)] pub struct bz_ctx { _p: [u8; 0] }
#[repr(C)] pub struct bz_params { _p: [u8; 0] }
#[repr(C)] pub struct bz_pk { _p: [u8; 0] }
#[repr(C)] pub struct bz_vk { _p: [u8; 0] }
#[repr(C)] pub struct bz_ipa { _p: [u8; 0] }
/// all-gather callback of bz_ctx_set_sharding: gather `bytes_per_rank` bytes of every rank's send buffer into the receive buffer
pub type bz_allgather_fn = Option<unsafe extern "C" fn(user: *mut c_void, bytes_per_rank: usize) -> c_int>;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct bz_token { pub op: u32, pub a: u32, pub b: i32 }

#[repr(C)]
pub struct bz_circuit {
    pub k: u32, pub num_advice: u32, pub num_fixed: u32, pub num_instance: u32, pub degree: u32, pub blinding_factors: u32,
    pub n_advice_queries: u32, pub advice_queries: *const i32,
    pub n_fixed_queries: u32, pub fixed_queries: *const i32,
    pub n_instance_queries: u32, pub instance_queries: *const i32,
    pub n_perm_columns: u32, pub perm_columns: *const u32,
    pub n_constants: u32, pub constants: *const c_void,
    pub n_tokens: u32, pub tokens: *const bz_token,
    pub n_gate_polys: u32, pub gate_poly_offsets: *const u32,
    pub n_lookups: u32, pub lookup_input_counts: *const u32, pub lookup_table_counts: *const u32,
    pub lookup_expr_offsets: *const u32,
    pub vk_transcript_repr: [u8; 32],
}

pub const BZ_ERR_SYNTHESIS: c_int = -4;
pub const FIELD_FP: c_int = 0;
pub const FIELD_FQ: c_int = 1;
pub const CURVE_VESTA: c_int = 0;

/// Error of a failed call: the status code and `bz_last_error`'s text.
#[derive(Debug)]
pub struct BzError { pub code: c_int, pub msg: String }

fn check(ctx: *mut bz_ctx, rc: c_int) -> Result<(), BzError> {
    if rc == 0 { return Ok(()); }
    let msg = unsafe { std::ffi::CStr::from_ptr(bz_last_error(ctx)).to_string_lossy().into_owned() };
    Err(BzError { code: rc, msg })
}

thread_local! { static CTX: RefCell<*mut bz_ctx> = RefCell::new(std::ptr::null_mut()); }

/// One context per thread on the GPU `BZ_DEVICE` names (default 0); a context may be used by one thread at a time (bzhalo2.h).
pub fn ctx() -> *mut bz_ctx {
    CTX.with(|c| {
        let mut c = c.borrow_mut();
        if c.is_null() {
            let dev = std::env::var("BZ_DEVICE").ok().and_then(|s| s.parse().ok()).unwrap_or(0);
            let rc = unsafe { bz_ctx_create(dev, std::ptr::null_mut(), &mut *c) };
            assert_eq!(rc, 0, "bz_ctx_create failed: no CUDA device (libbzhalo2 has no CPU fallback)");
        }
        *c
    })
}

// ---- marshalling --------------------------------------------------------------------------------------------------
/// x || y in memory (Montgomery) form; the identity becomes 64 zero bytes.
pub fn affine_to_bytes<C: CurveAffine>(p: &C) -> [u8; 64] where C::Base: Copy {
    let mut out = [0u8; 64];
    if let Some(c) = Option::<pasta_curves::arithmetic::Coordinates<C>>::from(p.coordinates()) {
        unsafe {
            out[..32].copy_from_slice(std::slice::from_raw_parts(c.x() as *const C::Base as *const u8, 32));
            out[32..].copy_from_slice(std::slice::from_raw_parts(c.y() as *const C::Base as *const u8, 32));
        }
    }
    out
}
pub fn affine_from_bytes(b: &[u8; 64]) -> vesta::Affine {
    if b.iter().all(|v| *v == 0) { return vesta::Affine::identity(); }
    let (mut x, mut y) = (Fq::zero(), Fq::zero());
    unsafe {
        std::ptr::copy_nonoverlapping(b.as_ptr(), &mut x as *mut Fq as *mut u8, 32);
        std::ptr::copy_nonoverlapping(b.as_ptr().add(32), &mut y as *mut Fq as *mut u8, 32);
    }
    vesta::Affine::from_xy(x, y).unwrap()
}
fn flatten_points(bases: &[vesta::Affine]) -> Vec<u8> {
    let mut flat = vec![0u8; bases.len() * 64];
    for (i, b) in bases.iter().enumerate() { flat[i * 64..(i + 1) * 64].copy_from_slice(&affine_to_bytes(b)); }
    flat
}

// ---- arithmetic.rs / poly/domain.rs -----------------------------------------------------------------------------------
/// `arithmetic::best_multiexp::<vesta::Affine>`
pub fn best_multiexp(coeffs: &[Fp], bases: &[vesta::Affine]) -> Result<vesta::Point, BzError> {
    assert_eq!(coeffs.len(), bases.len());
    let flat = flatten_points(bases);
    let mut jac = [Fq::zero(); 3];
    let c = ctx();
    check(c, unsafe { bz_best_multiexp(c, CURVE_VESTA, coeffs.as_ptr() as *const c_void, flat.as_ptr() as *const c_void, coeffs.len() as u64, jac.as_mut_ptr() as *mut c_void) })?;
    Ok(vesta::Point::new_jacobian(jac[0], jac[1], jac[2]).unwrap())
}
/// `arithmetic::best_fft` over field elements (omega must be the domain generator or its inverse: all halo2_proofs passes)
pub fn best_fft(a: &mut [Fp], omega: Fp, log_n: u32) -> Result<(), BzError> {
    let c = ctx();
    check(c, unsafe { bz_best_fft(c, FIELD_FP, a.as_mut_ptr() as *mut c_void, &omega as *const Fp as *const c_void, log_n) })
}
pub fn lagrange_to_coeff(a: &mut [Fp], k: u32) -> Result<(), BzError> {
    let c = ctx();
    check(c, unsafe { bz_lagrange_to_coeff(c, FIELD_FP, a.as_mut_ptr() as *mut c_void, k) })
}
pub fn coeff_to_extended(coeffs: &[Fp], k: u32, extended_k: u32) -> Result<Vec<Fp>, BzError> {
    let mut out = vec![Fp::zero(); 1 << extended_k];
    let c = ctx();
    check(c, unsafe { bz_coeff_to_extended(c, FIELD_FP, coeffs.as_ptr() as *const c_void, out.as_mut_ptr() as *mut c_void, k, extended_k) })?;
    Ok(out)
}
pub fn extended_to_coeff(a: &mut [Fp], extended_k: u32) -> Result<(), BzError> {
    let c = ctx();
    check(c, unsafe { bz_extended_to_coeff(c, FIELD_FP, a.as_mut_ptr() as *mut c_void, extended_k) })
}
pub fn divide_by_vanishing_poly(a: &mut [Fp], k: u32, extended_k: u32) -> Result<(), BzError> {
    let c = ctx();
    check(c, unsafe { bz_divide_by_vanishing(c, FIELD_FP, k, extended_k, a.as_mut_ptr() as *mut c_void) })
}
/// `arithmetic::eval_polynomial` for many (polynomial, point) pairs
pub fn eval_many(polys: &[&[Fp]], points: &[Fp]) -> Result<Vec<Fp>, BzError> {
    assert_eq!(polys.len(), points.len());
    let ptrs: Vec<*const c_void> = polys.iter().map(|p| p.as_ptr() as *const c_void).collect();
    let mut out = vec![Fp::zero(); polys.len()];
    let c = ctx();
    let n = polys.first().map(|p| p.len()).unwrap_or(0) as u64;
    check(c, unsafe { bz_eval_many(c, FIELD_FP, n, polys.len() as u32, ptrs.as_ptr(), points.as_ptr() as *const c_void, out.as_mut_ptr() as *mut c_void) })?;
    Ok(out)
}
/// `arithmetic::kate_division`
pub fn kate_division(a: &[Fp], point: Fp) -> Result<Vec<Fp>, BzError> {
    let mut q = vec![Fp::zero(); a.len() - 1];
    let c = ctx();
    check(c, unsafe { bz_kate_div(c, FIELD_FP, a.len() as u64, a.as_ptr() as *const c_void, &point as *const Fp as *const c_void, q.as_mut_ptr() as *mut c_void) })?;
    Ok(q)
}
/// acc = acc * x + poly
pub fn axpy(acc: &mut [Fp], x: Fp, poly: &[Fp]) -> Result<(), BzError> {
    assert_eq!(acc.len(), poly.len());
    let c = ctx();
    check(c, unsafe { bz_axpy(c, FIELD_FP, acc.len() as u64, acc.as_mut_ptr() as *mut c_void, &x as *const Fp as *const c_void, poly.as_ptr() as *const c_void) })
}
/// one column set of `permutation::Argument::commit`
#[allow(clippy::too_many_arguments)]
pub fn perm_product(k: u32, values: &[&[Fp]], sigmas: &[&[Fp]], beta: Fp, gamma: Fp, delta_omega0: Fp, z0: Fp) -> Result<Vec<Fp>, BzError> {
    assert_eq!(values.len(), sigmas.len());
    let v: Vec<*const c_void> = values.iter().map(|p| p.as_ptr() as *const c_void).collect();
    let s: Vec<*const c_void> = sigmas.iter().map(|p| p.as_ptr() as *const c_void).collect();
    let mut z = vec![Fp::zero(); 1 << k];
    let c = ctx();
    let p = |x: &Fp| x as *const Fp as *const c_void;
    check(c, unsafe { bz_perm_product(c, FIELD_FP, k, v.len() as u32, v.as_ptr(), s.as_ptr(), p(&beta), p(&gamma), p(&delta_omega0), p(&z0), z.as_mut_ptr() as *mut c_void) })?;
    Ok(z)
}
/// `lookup::permute_expression_pair`; `Err(code == BZ_ERR_SYNTHESIS)` maps to `Error::ConstraintSystemFailure`
pub fn lookup_permute(k: u32, usable_rows: u32, input: &[Fp], table: &[Fp]) -> Result<(Vec<Fp>, Vec<Fp>), BzError> {
    let (mut a, mut s) = (vec![Fp::zero(); 1 << k], vec![Fp::zero(); 1 << k]);
    let c = ctx();
    check(c, unsafe { bz_lookup_permute(c, FIELD_FP, k, usable_rows, input.as_ptr() as *const c_void, table.as_ptr() as *const c_void, a.as_mut_ptr() as *mut c_void, s.as_mut_ptr() as *mut c_void) })?;
    Ok((a, s))
}
#[allow(clippy::too_many_arguments)]
pub fn lookup_product(k: u32, input: &[Fp], table: &[Fp], permuted_input: &[Fp], permuted_table: &[Fp], beta: Fp, gamma: Fp) -> Result<Vec<Fp>, BzError> {
    let mut z = vec![Fp::zero(); 1 << k];
    let c = ctx();
    let p = |x: &[Fp]| x.as_ptr() as *const c_void;
    check(c, unsafe { bz_lookup_product(c, FIELD_FP, k, p(input), p(table), p(permuted_input), p(permuted_table), &beta as *const Fp as *const c_void, &gamma as *const Fp as *const c_void, z.as_mut_ptr() as *mut c_void) })?;
    Ok(z)
}

// ---- Params / ProvingKey handles ----------------------------------------------------------------------------------------
pub struct DeviceParams(pub *mut bz_params);
unsafe impl Send for DeviceParams {}
unsafe impl Sync for DeviceParams {}
impl Drop for DeviceParams { fn drop(&mut self) { unsafe { bz_params_destroy(self.0) } } }
impl DeviceParams {
    /// from the four fields of `Params<vesta::Affine>`
    pub fn new(k: u32, g: &[vesta::Affine], g_lagrange: &[vesta::Affine], w: &vesta::Affine, u: &vesta::Affine) -> Result<Self, BzError> {
        let (fg, fl) = (flatten_points(g), flatten_points(g_lagrange));
        let (w, u) = (affine_to_bytes(w), affine_to_bytes(u));
        let mut h = std::ptr::null_mut();
        let c = ctx();
        check(c, unsafe { bz_params_create(c, k, CURVE_VESTA, fg.as_ptr() as *const c_void, fl.as_ptr() as *const c_void, w.as_ptr() as *const c_void, u.as_ptr() as *const c_void, 0, &mut h) })?;
        Ok(DeviceParams(h))
    }
    /// `Params::commit` (lagrange = false) / `Params::commit_lagrange` (true), already normalised
    pub fn commit(&self, lagrange: bool, poly: &[Fp], blind: Fp) -> Result<vesta::Affine, BzError> {
        let mut out = [0u8; 64];
        let c = ctx();
        check(c, unsafe { bz_params_commit(c, self.0, lagrange as c_int, poly.as_ptr() as *const c_void, &blind as *const Fp as *const c_void, out.as_mut_ptr() as *mut c_void) })?;
        Ok(affine_from_bytes(&out))
    }
}
/// `Params::new(k)` computed on the device: (g, g_lagrange, w, u)
pub fn params_new(k: u32) -> Result<(Vec<vesta::Affine>, Vec<vesta::Affine>, vesta::Affine, vesta::Affine), BzError> {
    let n = 1usize << k;
    let (mut g, mut gl, mut w, mut u) = (vec![0u8; n * 64], vec![0u8; n * 64], [0u8; 64], [0u8; 64]);
    let c = ctx();
    check(c, unsafe { bz_params_new(c, k, CURVE_VESTA, g.as_mut_ptr() as *mut c_void, gl.as_mut_ptr() as *mut c_void, w.as_mut_ptr() as *mut c_void, u.as_mut_ptr() as *mut c_void) })?;
    let conv = |b: &[u8]| b.chunks_exact(64).map(|c| affine_from_bytes(c.try_into().unwrap())).collect::<Vec<_>>();
    Ok((conv(&g), conv(&gl), affine_from_bytes(&w), affine_from_bytes(&u)))
}

pub struct DevicePk(pub *mut bz_pk);
unsafe impl Send for DevicePk {}
unsafe impl Sync for DevicePk {}
impl Drop for DevicePk { fn drop(&mut self) { unsafe { bz_pk_destroy(self.0) } } }

/// `pk.vk.cs` flattened to the IR of SURVEY App. G.  The fork's `plonk/circuit.rs` implements `FlatCs::from(&ConstraintSystem)`
/// with crate-private access (expression trees -> postfix tokens: 0 Constant(index into `constants`), 1 Advice, 2 Fixed,
/// 3 Instance, 4 Negated, 5 Sum, 6 Product, 7 Scaled(index into `constants`); `Expression::Selector` cannot occur after
/// `compress_selectors`).
#[derive(Default)]
pub struct FlatCs {
    pub k: u32, pub num_advice: u32, pub num_fixed: u32, pub num_instance: u32, pub degree: u32, pub blinding_factors: u32,
    pub advice_queries: Vec<i32>, pub fixed_queries: Vec<i32>, pub instance_queries: Vec<i32>,   // (column, rotation) pairs
    pub perm_columns: Vec<u32>,                                                                   // (kind, index) pairs
    pub constants: Vec<Fp>, pub tokens: Vec<bz_token>, pub gate_poly_offsets: Vec<u32>,
    pub lookup_input_counts: Vec<u32>, pub lookup_table_counts: Vec<u32>, pub lookup_expr_offsets: Vec<u32>,
    pub vk_transcript_repr: [u8; 32],
}
impl FlatCs {
    pub fn as_ffi(&self) -> bz_circuit {
        bz_circuit {
            k: self.k, num_advice: self.num_advice, num_fixed: self.num_fixed, num_instance: self.num_instance, degree: self.degree,
            blinding_factors: self.blinding_factors,
            n_advice_queries: (self.advice_queries.len() / 2) as u32, advice_queries: self.advice_queries.as_ptr(),
            n_fixed_queries: (self.fixed_queries.len() / 2) as u32, fixed_queries: self.fixed_queries.as_ptr(),
            n_instance_queries: (self.instance_queries.len() / 2) as u32, instance_queries: self.instance_queries.as_ptr(),
            n_perm_columns: (self.perm_columns.len() / 2) as u32, perm_columns: self.perm_columns.as_ptr(),
            n_constants: self.constants.len() as u32, constants: self.constants.as_ptr() as *const c_void,
            n_tokens: self.tokens.len() as u32, tokens: self.tokens.as_ptr(),
            n_gate_polys: (self.gate_poly_offsets.len() - 1) as u32, gate_poly_offsets: self.gate_poly_offsets.as_ptr(),
            n_lookups: self.lookup_input_counts.len() as u32, lookup_input_counts: self.lookup_input_counts.as_ptr(),
            lookup_table_counts: self.lookup_table_counts.as_ptr(), lookup_expr_offsets: self.lookup_expr_offsets.as_ptr(),
            vk_transcript_repr: self.vk_transcript_repr,
        }
    }
}
impl DevicePk {
    /// `fixed_values`: num_fixed x n, `sigma_values`: n_perm_columns x n (pk.permutation.permutations), both Lagrange
    pub fn new(params: &DeviceParams, cs: &FlatCs, fixed_values: &[Fp], sigma_values: &[Fp]) -> Result<Self, BzError> {
        let mut h = std::ptr::null_mut();
        let c = ctx();
        let ffi = cs.as_ffi();
        check(c, unsafe { bz_pk_create(c, params.0, &ffi, fixed_values.as_ptr() as *const c_void, sigma_values.as_ptr() as *const c_void, &mut h) })?;
        Ok(DevicePk(h))
    }
    pub fn num_random(&self) -> usize { unsafe { bz_pk_num_random(self.0) as usize } }
    pub fn proof_size(&self) -> usize { unsafe { bz_pk_proof_size(self.0) as usize } }
}

/// `VerifyingKey` on the device: the flattened `vk.cs`, `vk.fixed_commitments` and the permutation commitments.  No fixed values
/// and no sigma columns; creating it allocates no device memory.  `params` must outlive it.
pub struct DeviceVk(pub *mut bz_vk);
unsafe impl Send for DeviceVk {}
unsafe impl Sync for DeviceVk {}
impl Drop for DeviceVk { fn drop(&mut self) { unsafe { bz_vk_destroy(self.0) } } }
impl DeviceVk {
    pub fn new(params: &DeviceParams, cs: &FlatCs, fixed_commitments: &[vesta::Affine], perm_commitments: &[vesta::Affine]) -> Result<Self, BzError> {
        let (fc, pc) = (flatten_points(fixed_commitments), flatten_points(perm_commitments));
        let mut h = std::ptr::null_mut();
        let c = ctx();
        let ffi = cs.as_ffi();
        check(c, unsafe { bz_vk_create(c, params.0, &ffi, fc.as_ptr() as *const c_void, pc.as_ptr() as *const c_void, &mut h) })?;
        Ok(DeviceVk(h))
    }
    pub fn proof_size(&self) -> usize { unsafe { bz_vk_proof_size(self.0) as usize } }
}

// ---- create_proof / verify_proof ------------------------------------------------------------------------------------------
/// Pre-draw the RNG words `create_proof` consumes, in protocol order (`bz_pk_num_random` is shape-only).  `Fp::random(rng)` is
/// `from_u512` of eight `next_u64()` little-endian limbs (ff 0.12 `Field::random` for pasta); the device performs the same
/// reduction on the raw 64 bytes, so the same `RngCore` yields the proof stock halo2 would write.
pub fn predraw<R: RngCore>(rng: &mut R, n: usize) -> Vec<u8> {
    let mut out = vec![0u8; n * 64];
    for chunk in out.chunks_exact_mut(8) { chunk.copy_from_slice(&rng.next_u64().to_le_bytes()); }
    out
}

/// One call for `batch` proofs of one circuit: instances[b][col] values, advice[b] = num_advice x n scalars.  Returns the
/// proof byte strings exactly as `Blake2bWrite::finalize()` yields them in halo2_proofs 0.2.0.
pub fn create_proofs<R: RngCore>(pk: &DevicePk, instances: &[Vec<Vec<Fp>>], advice: &[Fp], rng: &mut R) -> Result<Vec<Vec<u8>>, BzError> {
    let batch = instances.len();
    let ncol = instances.first().map(|i| i.len()).unwrap_or(0);
    let lens: Vec<u32> = (0..ncol).map(|c| instances[0][c].len() as u32).collect();
    let stride = lens.iter().copied().max().unwrap_or(0).max(1);
    let mut inst = vec![Fp::zero(); batch * ncol * stride as usize];
    for (b, cols) in instances.iter().enumerate() {
        for (c, col) in cols.iter().enumerate() {
            assert_eq!(col.len() as u32, lens[c], "all proofs of a batch share the instance shape");
            inst[(b * ncol + c) * stride as usize..][..col.len()].copy_from_slice(col);
        }
    }
    let words = predraw(rng, pk.num_random() * batch);
    let size = pk.proof_size();
    let mut proofs = vec![0u8; size * batch];
    let c = ctx();
    check(c, unsafe { bz_create_proofs(c, pk.0, batch as u32, inst.as_ptr() as *const c_void, lens.as_ptr(), stride, advice.as_ptr() as *const c_void, words.as_ptr() as *const c_void, proofs.as_mut_ptr() as *mut c_void) })?;
    Ok(proofs.chunks_exact(size).map(|p| p.to_vec()).collect())
}

/// `verify_proof` with `SingleVerifier` semantics: one verdict per proof
pub fn verify_proofs(pk: &DevicePk, instances: &[Vec<Vec<Fp>>], proofs: &[Vec<u8>]) -> Result<Vec<bool>, BzError> {
    verify_with(instances, proofs, |c, batch, inst, lens, stride, flat, len, res| unsafe { bz_verify_proofs(c, pk.0, batch, inst, lens, stride, flat, len, res) })
}
/// The same from a verifying key alone (what `plonk::verify_proof` is given)
pub fn verify_proofs_vk(vk: &DeviceVk, instances: &[Vec<Vec<Fp>>], proofs: &[Vec<u8>]) -> Result<Vec<bool>, BzError> {
    verify_with(instances, proofs, |c, batch, inst, lens, stride, flat, len, res| unsafe { bz_verify_proofs_vk(c, vk.0, batch, inst, lens, stride, flat, len, res) })
}
/// packs the batch and calls `call(ctx, batch, instances, instance_lens, instance_stride, proofs, proof_len, results)`
fn verify_with(instances: &[Vec<Vec<Fp>>], proofs: &[Vec<u8>],
               call: impl Fn(*mut bz_ctx, u32, *const c_void, *const u32, u32, *const c_void, u32, *mut u8) -> c_int) -> Result<Vec<bool>, BzError> {
    let batch = proofs.len();
    let ncol = instances.first().map(|i| i.len()).unwrap_or(0);
    let lens: Vec<u32> = (0..ncol).map(|c| instances[0][c].len() as u32).collect();
    let stride = lens.iter().copied().max().unwrap_or(0).max(1);
    let mut inst = vec![Fp::zero(); batch * ncol * stride as usize];
    for (b, cols) in instances.iter().enumerate() {
        for (c, col) in cols.iter().enumerate() { inst[(b * ncol + c) * stride as usize..][..col.len()].copy_from_slice(col); }
    }
    let len = proofs.first().map(|p| p.len()).unwrap_or(0);
    let flat: Vec<u8> = proofs.iter().flat_map(|p| { assert_eq!(p.len(), len); p.iter().copied() }).collect();
    let mut res = vec![0u8; batch];
    let c = ctx();
    check(c, call(c, batch as u32, inst.as_ptr() as *const c_void, lens.as_ptr(), stride, flat.as_ptr() as *const c_void, len as u32, res.as_mut_ptr()))?;
    Ok(res.into_iter().map(|r| r == 1).collect())
}

/// The proof layout as a list of item kinds, in write order (SURVEY App. A): the fork's `create_proof` replays the device's
/// bytes into the caller's `TranscriptWrite` with it, so `transcript.finalize()` and the transcript's hash state are what
/// stock halo2 leaves behind.  Points are 32-byte compressed encodings, scalars 32-byte canonical little-endian.
#[derive(Clone, Copy, PartialEq, Eq, Debug)]
pub enum ProofItem { Point, Scalar }
#[allow(clippy::too_many_arguments)]
pub fn proof_layout(num_advice: usize, num_lookups: usize, num_perm_sets: usize, quotient_pieces: usize, num_evals: usize, num_point_sets: usize, k: usize) -> Vec<ProofItem> {
    use ProofItem::*;
    let mut v = Vec::new();
    v.extend(std::iter::repeat(Point).take(num_advice));                 // step 2
    v.extend(std::iter::repeat(Point).take(2 * num_lookups));            // step 5: A', S' per lookup
    v.extend(std::iter::repeat(Point).take(num_perm_sets));              // step 7
    v.extend(std::iter::repeat(Point).take(num_lookups));                // step 8
    v.push(Point);                                                       // step 9: random polynomial
    v.extend(std::iter::repeat(Point).take(quotient_pieces));            // step 12
    v.extend(std::iter::repeat(Scalar).take(num_evals));                 // steps 14-18
    v.push(Point);                                                       // step 20: q'
    v.extend(std::iter::repeat(Scalar).take(num_point_sets));            //          q_set(x3)
    v.push(Point);                                                       // step 21: S
    for _ in 0..k { v.push(Point); v.push(Point); }                      //          L_j, R_j
    v.push(Scalar); v.push(Scalar);                                      //          c, f
    v
}
/// `write_point` / `write_scalar` of every item of `proof` into `transcript` (any `TranscriptWrite<vesta::Affine, _>` whose
/// challenges are then discarded: the squeezes happened on the library's own Blake2b state).  The closure form keeps this crate
/// independent of halo2_proofs' traits; the fork passes `|p| transcript.write_point(p)` and `|s| transcript.write_scalar(s)`
/// and calls `squeeze_challenge` at the protocol's positions (the values equal the library's by construction).
pub fn replay_into(proof: &[u8], layout: &[ProofItem], mut write_point: impl FnMut(vesta::Affine) -> std::io::Result<()>,
                   mut write_scalar: impl FnMut(Fp) -> std::io::Result<()>) -> std::io::Result<()> {
    use group::GroupEncoding;
    assert_eq!(proof.len(), 32 * layout.len());
    for (item, bytes) in layout.iter().zip(proof.chunks_exact(32)) {
        let repr: [u8; 32] = bytes.try_into().unwrap();
        match item {
            ProofItem::Point => write_point(Option::from(vesta::Affine::from_bytes(&repr)).ok_or_else(|| std::io::Error::new(std::io::ErrorKind::Other, "invalid point in proof"))?)?,
            ProofItem::Scalar => write_scalar(Option::from(Fp::from_repr(repr)).ok_or_else(|| std::io::Error::new(std::io::ErrorKind::Other, "invalid scalar in proof"))?)?,
        }
    }
    Ok(())
}

// ---- poly/commitment/prover.rs: the folding loop --------------------------------------------------------------------------
pub struct Ipa(*mut bz_ipa);
impl Drop for Ipa { fn drop(&mut self) { if !self.0.is_null() { unsafe { bz_ipa_destroy(self.0) } } } }
impl Ipa {
    pub fn begin(params: &DeviceParams, p_prime: &[Fp], x3: Fp) -> Result<Self, BzError> {
        let mut h = std::ptr::null_mut();
        let c = ctx();
        check(c, unsafe { bz_ipa_begin(c, params.0, p_prime.as_ptr() as *const c_void, &x3 as *const Fp as *const c_void, &mut h) })?;
        Ok(Ipa(h))
    }
    pub fn round(&mut self, z: Fp, l_rand: Fp, r_rand: Fp) -> Result<(vesta::Affine, vesta::Affine), BzError> {
        let (mut l, mut r) = ([0u8; 64], [0u8; 64]);
        let c = ctx();
        let p = |x: &Fp| x as *const Fp as *const c_void;
        check(c, unsafe { bz_ipa_round(c, self.0, p(&z), p(&l_rand), p(&r_rand), l.as_mut_ptr() as *mut c_void, r.as_mut_ptr() as *mut c_void) })?;
        Ok((affine_from_bytes(&l), affine_from_bytes(&r)))
    }
    pub fn fold(&mut self, u: Fp) -> Result<(), BzError> {
        let u_inv = u.invert().unwrap();
        let c = ctx();
        check(c, unsafe { bz_ipa_fold(c, self.0, &u as *const Fp as *const c_void, &u_inv as *const Fp as *const c_void) })
    }
    pub fn finish(mut self) -> Result<Fp, BzError> {
        let mut out = Fp::zero();
        let c = ctx();
        let h = std::mem::replace(&mut self.0, std::ptr::null_mut());
        check(c, unsafe { bz_ipa_finish(c, h, &mut out as *mut Fp as *mut c_void) })?;
        Ok(out)
    }
}

// silence "unused" for items only the fork uses
#[allow(dead_code)]
fn _uses(_: Fq, _: &dyn Fn(vesta::Point) -> vesta::Affine) { let _ = <Fp as FieldExt>::ROOT_OF_UNITY; let _ = |p: vesta::Point| p.to_affine(); }
