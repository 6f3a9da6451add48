//! B200 batch engine behind the crate's own types (`--features b200`).
//!
//! This file is the reference-side binding of `include/decaf377_b200.h`: it lives at
//! `src/gpu.rs` of the decaf377 crate (v0.10.1, `arkworks` + default u64 backend), declared in
//! `src/lib.rs` as `#[cfg(feature = "b200")] pub mod gpu;`.  It adds *batch* forms of the hot
//! path next to the existing per-element API and keeps the crate's names and error
//! behaviour:
//!
//! | crate item (file:line)                                              | batch form here |
//! |---|---|
//! | `Encoding::vartime_decompress` (ark_curve/encoding.rs:32-83)        | `decompress_batch` |
//! | `Element::vartime_compress` (ark_curve/encoding.rs:116-128)         | `compress_batch` |
//! | `Element::encode_to_curve` / `hash_to_curve` (elligator.rs:67-76)   | `encode_to_curve_batch`, `hash_to_curve_batch`, `*_bytes` for raw hash output |
//! | `&Element * &Fr` (ark_curve/ops/projective.rs:106-191)              | `mul_batch` |
//! | `Element::GENERATOR * s` (element/projective.rs:20-22)              | `generator_mul_batch` |
//! | `Add / Sub / Neg` (ark_curve/ops/projective.rs:5-104), doubling     | `add_batch`, `sub_batch`, `neg_batch`, `double_batch` |
//! | `Element::vartime_multiscalar_mul` (element/projective.rs:99-117)   | `vartime_multiscalar_mul`, `vartime_multiscalar_mul_multi_gpu`, `vartime_multiscalar_mul_batch` (many small ones) |
//! | `VariableBaseMSM::msm` over long-lived bases (ark_curve/element.rs:27-37) | `GpuBases::new`, `GpuBases::msm` |
//! | `B * s` / `sum_j s_j * B_j` for long-lived bases B_j (fixed-base tables) | `GpuFixedBases::new`, `GpuFixedBases::mul`, `GpuFixedBases::mul_compressed` |
//! | `CurveGroup::normalize_batch` (ark_curve/element.rs:74-81)          | `normalize_batch` |
//! | `OnCurve::is_on_curve` (ark_curve/on_curve.rs:17-38)                | `is_on_curve_batch` |
//!
//! Wire formats (see the header): an `Element` travels as X‖Y‖Z‖T, four 32-byte
//! little-endian Montgomery limb strings -- exactly the `[u64; 4]` inside each coordinate,
//! so marshalling is a copy, not a conversion.  `Fr` scalars travel as their in-memory
//! Montgomery limbs as well (`D377_SCALARS_MONTGOMERY`); the GPU converts them.
//!
//! The only thing this module needs from the rest of the crate that v0.10.1 does not have is
//! the outbound limb accessor `to_montgomery_limbs` on `Fq` / `Fr` (the inbound direction,
//! `from_montgomery_limbs`, exists: fields/fq/u64/wrapper.rs:82, fr/u64/wrapper.rs:71).  It
//! is three lines per field; see `rust/patches/0001-b200-feature.patch`.
//!
//! There is no CPU fallback in here: every function returns `GpuError` when the library or
//! the GPU is missing, and callers keep using the per-element API in that case.

#![cfg(feature = "b200")]

extern crate alloc;
extern crate std;

use alloc::vec;
use alloc::vec::Vec;
use core::ffi::{c_char, c_int, c_void};
use std::ffi::CStr;

use crate::ark_curve::{AffinePoint, EdwardsAffine, EdwardsProjective};
use crate::{Element, Encoding, EncodingError, Fq, Fr};

// ---------------------------------------------------------------------------------------------
// include/decaf377_b200.h
// ---------------------------------------------------------------------------------------------
pub const D377_OK: c_int = 0;
pub const D377_ERR_INVALID_ARG: c_int = -1;
pub const D377_ERR_CUDA: c_int = -2;
pub const D377_ERR_NOT_INITIALISED: c_int = -3;
pub const D377_ERR_SCALAR_RANGE: c_int = -4;
pub const D377_ERR_INVALID_ENCODING: c_int = -5;

const PT_ELEMENT: c_int = 0;
const PT_ENCODING: c_int = 1;
const PT_AFFINE: c_int = 2;
const PT_BASES: c_int = 4;
const SCALARS_MONTGOMERY: c_int = 0x100;
const OUT_ELEMENT: c_int = 0;
const OUT_ENCODING: c_int = 1;

#[link(name = "decaf377_b200")]
extern "C" {
    fn d377_init(device: c_int) -> c_int;
    fn d377_init_multi(devices: *const c_int, ndev: c_int) -> c_int;
    fn d377_set_device(device: c_int) -> c_int;
    fn d377_shutdown() -> c_int;
    fn d377_last_error() -> *const c_char;

    fn d377_batch_decompress(enc: *const u8, n: usize, elements: *mut u8, ok: *mut u8) -> c_int;
    fn d377_batch_compress(elements: *const u8, n: usize, enc: *mut u8) -> c_int;
    fn d377_batch_decompress_fmt(enc: *const u8, n: usize, out_format: c_int, out: *mut u8, ok: *mut u8) -> c_int;
    fn d377_batch_compress_fmt(points: *const u8, point_format: c_int, n: usize, enc: *mut u8) -> c_int;
    fn d377_batch_encode_to_curve_wide(r: *const u8, in_width: usize, n: usize, out: *mut u8, out_format: c_int) -> c_int;
    fn d377_batch_hash_to_curve_wide(r1: *const u8, r2: *const u8, in_width: usize, n: usize, out: *mut u8, out_format: c_int) -> c_int;
    fn d377_batch_scalar_mul(points: *const u8, point_format: c_int, scalars: *const u8, n: usize,
                             out: *mut u8, out_format: c_int, ok: *mut u8) -> c_int;
    fn d377_fixed_base_mul(scalars: *const u8, n: usize, out: *mut u8, out_format: c_int) -> c_int;
    fn d377_batch_add(a: *const u8, b: *const u8, n: usize, out: *mut u8) -> c_int;
    fn d377_batch_sub(a: *const u8, b: *const u8, n: usize, out: *mut u8) -> c_int;
    fn d377_batch_neg(a: *const u8, n: usize, out: *mut u8) -> c_int;
    fn d377_batch_double(a: *const u8, n: usize, out: *mut u8) -> c_int;
    fn d377_batch_on_curve(elements: *const u8, n: usize, check_order: c_int, ok: *mut u8) -> c_int;
    fn d377_batch_normalize(elements: *const u8, n: usize, affine: *mut u8) -> c_int;
    fn d377_msm(scalars: *const u8, points: *const u8, point_format: c_int, n: usize,
                out_element: *mut u8, out_encoding: *mut u8) -> c_int;
    fn d377_msm_multi(scalars: *const u8, points: *const u8, point_format: c_int, n: usize, ngpu: c_int,
                      out_element: *mut u8, out_encoding: *mut u8) -> c_int;
    fn d377_batch_msm(scalars: *const u8, points: *const u8, point_format: c_int, offsets: *const u32, nmsm: usize,
                      out: *mut u8, out_format: c_int, ok: *mut u8) -> c_int;
    fn d377_msm_segmented(scalars: *const u8, points: *const u8, point_format: c_int, offsets: *const u32,
                          nmsm: usize, out: *mut u8, out_format: c_int, ok: *mut u8) -> c_int;
    fn d377_msm_bases_create(points: *const u8, point_format: c_int, n: usize, bases: *mut *mut u8) -> c_int;
    fn d377_msm_bases_destroy(bases: *mut u8) -> c_int;
    fn d377_msm_bases_create_windowed(points: *const u8, point_format: c_int, n: usize, c: c_int,
                                      bases: *mut *mut u8) -> c_int;
    fn d377_msm_bases_create_windowed_dev(points: *const u8, point_format: c_int, n: usize, c: c_int,
                                          bases: *mut *mut u8) -> c_int;
    fn d377_msm_bases_info(bases: *const u8, n: *mut usize, c: *mut c_int, windows: *mut c_int,
                           bytes: *mut usize) -> c_int;
    fn d377_fixed_bases_create(points: *const u8, point_format: c_int, k: usize, tables: *mut *mut u8) -> c_int;
    fn d377_fixed_bases_destroy(tables: *mut u8) -> c_int;
    fn d377_fixed_bases_mul(tables: *const u8, scalars: *const u8, n: usize, out: *mut u8, out_format: c_int) -> c_int;
    fn d377_host_alloc(bytes: usize) -> *mut c_void;
    fn d377_host_free(p: *mut c_void) -> c_int;
}

/// Failure of the GPU path (never a failure of a single element: those are `EncodingError`s
/// inside the returned vectors, as in the per-element API).
#[derive(Debug, Clone)]
pub struct GpuError {
    pub code: i32,
    pub message: alloc::string::String,
}

impl core::fmt::Display for GpuError {
    fn fmt(&self, f: &mut core::fmt::Formatter<'_>) -> core::fmt::Result {
        write!(f, "decaf377_b200 error {}: {}", self.code, self.message)
    }
}

impl std::error::Error for GpuError {}

fn check(rc: c_int) -> Result<(), GpuError> {
    if rc == D377_OK {
        return Ok(());
    }
    // SAFETY: d377_last_error returns a NUL-terminated string owned by the library
    // (thread-local storage), valid until this thread's next call into it.
    let message = unsafe { CStr::from_ptr(d377_last_error()) }.to_string_lossy().into_owned();
    Err(GpuError { code: rc, message })
}

/// `d377_init`: create the engine of one GPU and make it the process default.
pub fn init(device: i32) -> Result<(), GpuError> {
    check(unsafe { d377_init(device) })
}

/// `d377_init_multi`: engines for several GPUs of the box (`vartime_multiscalar_mul_multi_gpu`).
pub fn init_multi(devices: &[i32]) -> Result<(), GpuError> {
    check(unsafe { d377_init_multi(devices.as_ptr(), devices.len() as c_int) })
}

/// `d377_set_device`: the initialised GPU this *thread's* calls act on (e.g. one rayon worker
/// per GPU); a negative value returns to the process default.
pub fn set_device(device: i32) -> Result<(), GpuError> {
    check(unsafe { d377_set_device(device) })
}

pub fn shutdown() -> Result<(), GpuError> {
    check(unsafe { d377_shutdown() })
}

// ---------------------------------------------------------------------------------------------
// marshalling: the crate's types <-> the wire images of the header
// ---------------------------------------------------------------------------------------------
#[inline]
fn put_limbs(out: &mut [u8], limbs: [u64; 4]) {
    for (i, l) in limbs.iter().enumerate() {
        out[8 * i..8 * i + 8].copy_from_slice(&l.to_le_bytes());
    }
}

#[inline]
fn get_limbs(b: &[u8]) -> [u64; 4] {
    let mut l = [0u64; 4];
    for i in 0..4 {
        let mut w = [0u8; 8];
        w.copy_from_slice(&b[8 * i..8 * i + 8]);
        l[i] = u64::from_le_bytes(w);
    }
    l
}

/// X‖Y‖Z‖T, each the 32 little-endian bytes of the coordinate's Montgomery limbs
/// (`Projective` is not `repr(C)` and orders its fields x, y, t, z: copy field by field).
#[inline]
fn element_to_wire(e: &Element, out: &mut [u8]) {
    put_limbs(&mut out[0..32], e.inner.x.to_montgomery_limbs());
    put_limbs(&mut out[32..64], e.inner.y.to_montgomery_limbs());
    put_limbs(&mut out[64..96], e.inner.z.to_montgomery_limbs());
    put_limbs(&mut out[96..128], e.inner.t.to_montgomery_limbs());
}

/// The library writes canonical Montgomery limbs (< q), which is what `from_montgomery_limbs`
/// (fields/fq/u64/wrapper.rs:82, `new_unchecked`) expects.
#[inline]
fn wire_to_element(b: &[u8]) -> Element {
    let x = Fq::from_montgomery_limbs(get_limbs(&b[0..32]));
    let y = Fq::from_montgomery_limbs(get_limbs(&b[32..64]));
    let z = Fq::from_montgomery_limbs(get_limbs(&b[64..96]));
    let t = Fq::from_montgomery_limbs(get_limbs(&b[96..128]));
    Element { inner: EdwardsProjective::new_unchecked(x, y, t, z) }
}

#[inline]
fn wire_to_affine(b: &[u8]) -> AffinePoint {
    let x = Fq::from_montgomery_limbs(get_limbs(&b[0..32]));
    let y = Fq::from_montgomery_limbs(get_limbs(&b[32..64]));
    AffinePoint { inner: EdwardsAffine::new_unchecked(x, y) }
}

fn elements_to_wire(els: &[Element]) -> Vec<u8> {
    let mut w = vec![0u8; 128 * els.len()];
    for (e, chunk) in els.iter().zip(w.chunks_exact_mut(128)) {
        element_to_wire(e, chunk);
    }
    w
}

fn wire_to_elements(w: &[u8]) -> Vec<Element> {
    w.chunks_exact(128).map(wire_to_element).collect()
}

/// In-memory Montgomery limbs of the scalars (`D377_SCALARS_MONTGOMERY`): no
/// `Fr::to_bytes` (a Montgomery reduction per scalar) on the host.
fn scalars_to_wire(sc: &[Fr]) -> Vec<u8> {
    let mut w = vec![0u8; 32 * sc.len()];
    for (s, chunk) in sc.iter().zip(w.chunks_exact_mut(32)) {
        put_limbs(chunk, s.to_montgomery_limbs());
    }
    w
}

/// Canonical little-endian bytes of field elements (`Fq::to_bytes`): the input of the
/// Elligator entry points, which reduce whatever bytes they get exactly like
/// `Fq::from_le_bytes_mod_order` (fields/fq.rs:90-102).
fn fq_to_canonical(r: &[Fq]) -> Vec<u8> {
    let mut w = vec![0u8; 32 * r.len()];
    for (x, chunk) in r.iter().zip(w.chunks_exact_mut(32)) {
        chunk.copy_from_slice(&x.to_bytes());
    }
    w
}

fn encodings_to_wire(encs: &[Encoding]) -> Vec<u8> {
    let mut w = vec![0u8; 32 * encs.len()];
    for (e, chunk) in encs.iter().zip(w.chunks_exact_mut(32)) {
        chunk.copy_from_slice(&e.0);
    }
    w
}

fn wire_to_encodings(w: &[u8]) -> Vec<Encoding> {
    w.chunks_exact(32)
        .map(|c| {
            let mut b = [0u8; 32];
            b.copy_from_slice(c);
            Encoding(b)
        })
        .collect()
}

// ---------------------------------------------------------------------------------------------
// batch codec
// ---------------------------------------------------------------------------------------------

/// `Encoding::vartime_decompress` over a slice: one `Result` per encoding, `InvalidEncoding`
/// for exactly the inputs the per-element call rejects.
pub fn decompress_batch(encs: &[Encoding]) -> Result<Vec<Result<Element, EncodingError>>, GpuError> {
    let n = encs.len();
    let inp = encodings_to_wire(encs);
    let mut out = vec![0u8; 128 * n];
    let mut ok = vec![0u8; n];
    check(unsafe { d377_batch_decompress(inp.as_ptr(), n, out.as_mut_ptr(), ok.as_mut_ptr()) })?;
    Ok(out
        .chunks_exact(128)
        .zip(ok.iter())
        .map(|(w, &good)| if good == 1 { Ok(wire_to_element(w)) } else { Err(EncodingError::InvalidEncoding) })
        .collect())
}

/// `Element::vartime_compress` over a slice.
pub fn compress_batch(els: &[Element]) -> Result<Vec<Encoding>, GpuError> {
    let n = els.len();
    let inp = elements_to_wire(els);
    let mut out = vec![0u8; 32 * n];
    check(unsafe { d377_batch_compress(inp.as_ptr(), n, out.as_mut_ptr()) })?;
    Ok(wire_to_encodings(&out))
}

/// `CanonicalSerialize for AffinePoint` (ark_curve/serialize.rs:30-46) over a slice: the
/// 64-byte affine image goes to the GPU as it is, no `Element` is built on the host.
pub fn serialize_affine_batch(pts: &[AffinePoint]) -> Result<Vec<Encoding>, GpuError> {
    let n = pts.len();
    let mut inp = vec![0u8; 64 * n];
    for (p, chunk) in pts.iter().zip(inp.chunks_exact_mut(64)) {
        put_limbs(&mut chunk[0..32], p.inner.x.to_montgomery_limbs());
        put_limbs(&mut chunk[32..64], p.inner.y.to_montgomery_limbs());
    }
    let mut out = vec![0u8; 32 * n];
    check(unsafe { d377_batch_compress_fmt(inp.as_ptr(), PT_AFFINE, n, out.as_mut_ptr()) })?;
    Ok(wire_to_encodings(&out))
}

/// `CanonicalDeserialize for AffinePoint` (ark_curve/serialize.rs:8-28) over a slice:
/// `SerializationError::InvalidData` per element becomes `Err(InvalidEncoding)`.
pub fn deserialize_affine_batch(encs: &[Encoding]) -> Result<Vec<Result<AffinePoint, EncodingError>>, GpuError> {
    let n = encs.len();
    let inp = encodings_to_wire(encs);
    let mut out = vec![0u8; 64 * n];
    let mut ok = vec![0u8; n];
    check(unsafe { d377_batch_decompress_fmt(inp.as_ptr(), n, PT_AFFINE, out.as_mut_ptr(), ok.as_mut_ptr()) })?;
    Ok(out
        .chunks_exact(64)
        .zip(ok.iter())
        .map(|(w, &good)| if good == 1 { Ok(wire_to_affine(w)) } else { Err(EncodingError::InvalidEncoding) })
        .collect())
}

/// `Element::encode_to_curve` over a slice of field elements.
pub fn encode_to_curve_batch(r: &[Fq]) -> Result<Vec<Element>, GpuError> {
    let n = r.len();
    let inp = fq_to_canonical(r);
    let mut out = vec![0u8; 128 * n];
    check(unsafe { d377_batch_encode_to_curve_wide(inp.as_ptr(), 32, n, out.as_mut_ptr(), OUT_ELEMENT) })?;
    Ok(wire_to_elements(&out))
}

/// `Element::encode_to_curve(&Fq::from_le_bytes_mod_order(chunk))` for every `width`-byte
/// chunk of `bytes` (e.g. 64-byte hash outputs), reduction included, on the GPU.
pub fn encode_to_curve_bytes(bytes: &[u8], width: usize) -> Result<Vec<Element>, GpuError> {
    assert!(width > 0 && bytes.len() % width == 0);
    let n = bytes.len() / width;
    let mut out = vec![0u8; 128 * n];
    check(unsafe { d377_batch_encode_to_curve_wide(bytes.as_ptr(), width, n, out.as_mut_ptr(), OUT_ELEMENT) })?;
    Ok(wire_to_elements(&out))
}

/// `Element::encode_to_curve(r).vartime_compress()` in one pass (one inverse square root
/// per element instead of two).
pub fn encode_to_curve_compressed_batch(r: &[Fq]) -> Result<Vec<Encoding>, GpuError> {
    let n = r.len();
    let inp = fq_to_canonical(r);
    let mut out = vec![0u8; 32 * n];
    check(unsafe { d377_batch_encode_to_curve_wide(inp.as_ptr(), 32, n, out.as_mut_ptr(), OUT_ENCODING) })?;
    Ok(wire_to_encodings(&out))
}

/// `Element::hash_to_curve` over two slices of equal length.
pub fn hash_to_curve_batch(r1: &[Fq], r2: &[Fq]) -> Result<Vec<Element>, GpuError> {
    let n = core::cmp::min(r1.len(), r2.len());
    let (a, b) = (fq_to_canonical(&r1[..n]), fq_to_canonical(&r2[..n]));
    let mut out = vec![0u8; 128 * n];
    check(unsafe { d377_batch_hash_to_curve_wide(a.as_ptr(), b.as_ptr(), 32, n, out.as_mut_ptr(), OUT_ELEMENT) })?;
    Ok(wire_to_elements(&out))
}

/// `hash_to_curve` from raw hash output: `r1`, `r2` hold `width` bytes per element.
pub fn hash_to_curve_bytes(r1: &[u8], r2: &[u8], width: usize) -> Result<Vec<Element>, GpuError> {
    assert!(width > 0 && r1.len() == r2.len() && r1.len() % width == 0);
    let n = r1.len() / width;
    let mut out = vec![0u8; 128 * n];
    check(unsafe { d377_batch_hash_to_curve_wide(r1.as_ptr(), r2.as_ptr(), width, n, out.as_mut_ptr(), OUT_ELEMENT) })?;
    Ok(wire_to_elements(&out))
}

// ---------------------------------------------------------------------------------------------
// group operations
// ---------------------------------------------------------------------------------------------
fn binop(f: unsafe extern "C" fn(*const u8, *const u8, usize, *mut u8) -> c_int, a: &[Element], b: &[Element])
         -> Result<Vec<Element>, GpuError> {
    let n = core::cmp::min(a.len(), b.len());
    let (wa, wb) = (elements_to_wire(&a[..n]), elements_to_wire(&b[..n]));
    let mut out = vec![0u8; 128 * n];
    check(unsafe { f(wa.as_ptr(), wb.as_ptr(), n, out.as_mut_ptr()) })?;
    Ok(wire_to_elements(&out))
}

fn unop(f: unsafe extern "C" fn(*const u8, usize, *mut u8) -> c_int, a: &[Element]) -> Result<Vec<Element>, GpuError> {
    let wa = elements_to_wire(a);
    let mut out = vec![0u8; 128 * a.len()];
    check(unsafe { f(wa.as_ptr(), a.len(), out.as_mut_ptr()) })?;
    Ok(wire_to_elements(&out))
}

/// `a[i] + b[i]` (ark_curve/ops/projective.rs:5-47).
pub fn add_batch(a: &[Element], b: &[Element]) -> Result<Vec<Element>, GpuError> {
    binop(d377_batch_add, a, b)
}

/// `a[i] - b[i]` (ark_curve/ops/projective.rs:50-87).
pub fn sub_batch(a: &[Element], b: &[Element]) -> Result<Vec<Element>, GpuError> {
    binop(d377_batch_sub, a, b)
}

/// `-a[i]` (ark_curve/ops/projective.rs:90-96).
pub fn neg_batch(a: &[Element]) -> Result<Vec<Element>, GpuError> {
    unop(d377_batch_neg, a)
}

/// `a[i] + a[i]`.
pub fn double_batch(a: &[Element]) -> Result<Vec<Element>, GpuError> {
    unop(d377_batch_double, a)
}

/// `scalars[i] * points[i]` (ark_curve/ops/projective.rs:106-191).
pub fn mul_batch(points: &[Element], scalars: &[Fr]) -> Result<Vec<Element>, GpuError> {
    let n = core::cmp::min(points.len(), scalars.len());
    let (wp, ws) = (elements_to_wire(&points[..n]), scalars_to_wire(&scalars[..n]));
    let mut out = vec![0u8; 128 * n];
    check(unsafe {
        d377_batch_scalar_mul(wp.as_ptr(), PT_ELEMENT | SCALARS_MONTGOMERY, ws.as_ptr(), n, out.as_mut_ptr(),
                              OUT_ELEMENT, core::ptr::null_mut())
    })?;
    Ok(wire_to_elements(&out))
}

/// The configuration-1 pipeline in one launch: `(s * E.vartime_decompress()?).vartime_compress()`
/// per element; an invalid encoding yields `Err(InvalidEncoding)` for that element only.
pub fn decompress_mul_compress_batch(encs: &[Encoding], scalars: &[Fr])
                                     -> Result<Vec<Result<Encoding, EncodingError>>, GpuError> {
    let n = core::cmp::min(encs.len(), scalars.len());
    let (we, ws) = (encodings_to_wire(&encs[..n]), scalars_to_wire(&scalars[..n]));
    let mut out = vec![0u8; 32 * n];
    let mut ok = vec![0u8; n];
    check(unsafe {
        d377_batch_scalar_mul(we.as_ptr(), PT_ENCODING | SCALARS_MONTGOMERY, ws.as_ptr(), n, out.as_mut_ptr(),
                              OUT_ENCODING, ok.as_mut_ptr())
    })?;
    Ok(wire_to_encodings(&out)
        .into_iter()
        .zip(ok.iter())
        .map(|(e, &good)| if good == 1 { Ok(e) } else { Err(EncodingError::InvalidEncoding) })
        .collect())
}

/// `Element::GENERATOR * s` for every scalar, over precomputed window tables.
pub fn generator_mul_batch(scalars: &[Fr]) -> Result<Vec<Element>, GpuError> {
    let ws = scalars_to_wire(scalars);
    let mut out = vec![0u8; 128 * scalars.len()];
    check(unsafe { d377_fixed_base_mul(ws.as_ptr(), scalars.len(), out.as_mut_ptr(), OUT_ELEMENT | SCALARS_MONTGOMERY) })?;
    Ok(wire_to_elements(&out))
}

/// `(Element::GENERATOR * s).vartime_compress()` for every scalar (no inverse square root:
/// the multiplication runs on the Jacobi quartic for large batches).
pub fn generator_mul_compressed_batch(scalars: &[Fr]) -> Result<Vec<Encoding>, GpuError> {
    let ws = scalars_to_wire(scalars);
    let mut out = vec![0u8; 32 * scalars.len()];
    check(unsafe { d377_fixed_base_mul(ws.as_ptr(), scalars.len(), out.as_mut_ptr(), OUT_ENCODING | SCALARS_MONTGOMERY) })?;
    Ok(wire_to_encodings(&out))
}

/// `CurveGroup::normalize_batch` / `ScalarMul::batch_convert_to_mul_base`
/// (ark_curve/element.rs:27-34,74-81).
pub fn normalize_batch(els: &[Element]) -> Result<Vec<AffinePoint>, GpuError> {
    let w = elements_to_wire(els);
    let mut out = vec![0u8; 64 * els.len()];
    check(unsafe { d377_batch_normalize(w.as_ptr(), els.len(), out.as_mut_ptr()) })?;
    Ok(out.chunks_exact(64).map(wire_to_affine).collect())
}

/// `OnCurve::is_on_curve` (ark_curve/on_curve.rs:17-38) for every element; `check_order`
/// includes the `[2r]P = 0` clause (one scalar multiplication per element).
pub fn is_on_curve_batch(els: &[Element], check_order: bool) -> Result<Vec<bool>, GpuError> {
    let w = elements_to_wire(els);
    let mut ok = vec![0u8; els.len()];
    check(unsafe { d377_batch_on_curve(w.as_ptr(), els.len(), check_order as c_int, ok.as_mut_ptr()) })?;
    Ok(ok.into_iter().map(|b| b == 1).collect())
}

// ---------------------------------------------------------------------------------------------
// Element::vartime_multiscalar_mul
// ---------------------------------------------------------------------------------------------

/// `Element::vartime_multiscalar_mul` (element/projective.rs:99-117) as a Pippenger MSM on
/// one GPU.  Like the crate's fold, the two sequences are zipped: the longer one is
/// truncated; an empty input gives `Element::default()`.
pub fn vartime_multiscalar_mul(scalars: &[Fr], points: &[Element]) -> Result<Element, GpuError> {
    let n = core::cmp::min(scalars.len(), points.len());
    let (ws, wp) = (scalars_to_wire(&scalars[..n]), elements_to_wire(&points[..n]));
    let mut out = [0u8; 128];
    check(unsafe {
        d377_msm(ws.as_ptr(), wp.as_ptr(), PT_ELEMENT | SCALARS_MONTGOMERY, n, out.as_mut_ptr(), core::ptr::null_mut())
    })?;
    Ok(wire_to_element(&out))
}

/// The same MSM cut into `ngpu` contiguous slices, one per GPU of `init_multi`; the 128-byte
/// partial sums meet on the first GPU (SURVEY 8e).
pub fn vartime_multiscalar_mul_multi_gpu(scalars: &[Fr], points: &[Element], ngpu: usize) -> Result<Element, GpuError> {
    let n = core::cmp::min(scalars.len(), points.len());
    let (ws, wp) = (scalars_to_wire(&scalars[..n]), elements_to_wire(&points[..n]));
    let mut out = [0u8; 128];
    check(unsafe {
        d377_msm_multi(ws.as_ptr(), wp.as_ptr(), PT_ELEMENT | SCALARS_MONTGOMERY, n, ngpu as c_int,
                       out.as_mut_ptr(), core::ptr::null_mut())
    })?;
    Ok(wire_to_element(&out))
}

/// The pairs of `jobs` back to back (Montgomery scalars, Element wire images) and the
/// segment offsets of the batch entry points.
fn pack_jobs(jobs: &[(&[Fr], &[Element])]) -> (Vec<u32>, Vec<u8>, Vec<u8>) {
    let mut offsets: Vec<u32> = Vec::with_capacity(jobs.len() + 1);
    offsets.push(0);
    let mut total = 0usize;
    for (s, p) in jobs {
        total += core::cmp::min(s.len(), p.len());
        offsets.push(total as u32);
    }
    let mut ws = vec![0u8; 32 * total];
    let mut wp = vec![0u8; 128 * total];
    let mut k = 0usize;
    for (s, p) in jobs {
        let n = core::cmp::min(s.len(), p.len());
        for i in 0..n {
            put_limbs(&mut ws[32 * k..32 * k + 32], s[i].to_montgomery_limbs());
            element_to_wire(&p[i], &mut wp[128 * k..128 * k + 128]);
            k += 1;
        }
    }
    (offsets, ws, wp)
}

/// Many independent `Element::vartime_multiscalar_mul` calls in one launch (e.g. a batch of
/// verification equations): `jobs[j]` is one (scalars, points) pair of slices, zipped like the
/// crate's fold.  Cost is per pair, not per job; see `d377_batch_msm`.
pub fn vartime_multiscalar_mul_batch(jobs: &[(&[Fr], &[Element])]) -> Result<Vec<Element>, GpuError> {
    let (offsets, ws, wp) = pack_jobs(jobs);
    let mut out = vec![0u8; 128 * jobs.len()];
    check(unsafe {
        d377_batch_msm(ws.as_ptr(), wp.as_ptr(), PT_ELEMENT | SCALARS_MONTGOMERY, offsets.as_ptr(), jobs.len(),
                       out.as_mut_ptr(), OUT_ELEMENT, core::ptr::null_mut())
    })?;
    Ok(wire_to_elements(&out))
}

/// The same results as `vartime_multiscalar_mul_batch`, from one segmented Pippenger over all
/// jobs (`d377_msm_segmented`): the cost is per pair and window plus per bucket instead of a
/// ladder per pair -- the call for many jobs of tens to tens of thousands of pairs.
pub fn vartime_multiscalar_mul_segmented(jobs: &[(&[Fr], &[Element])]) -> Result<Vec<Element>, GpuError> {
    let (offsets, ws, wp) = pack_jobs(jobs);
    let mut out = vec![0u8; 128 * jobs.len()];
    check(unsafe {
        d377_msm_segmented(ws.as_ptr(), wp.as_ptr(), PT_ELEMENT | SCALARS_MONTGOMERY, offsets.as_ptr(), jobs.len(),
                           out.as_mut_ptr(), OUT_ELEMENT, core::ptr::null_mut())
    })?;
    Ok(wire_to_elements(&out))
}

/// `<Element as VariableBaseMSM>::msm` over `AffinePoint` bases (ark_curve/element.rs:37).
pub fn msm_affine(bases: &[AffinePoint], scalars: &[Fr]) -> Result<Element, GpuError> {
    let n = core::cmp::min(scalars.len(), bases.len());
    let ws = scalars_to_wire(&scalars[..n]);
    let mut wp = vec![0u8; 64 * n];
    for (b, chunk) in bases[..n].iter().zip(wp.chunks_exact_mut(64)) {
        put_limbs(&mut chunk[0..32], b.inner.x.to_montgomery_limbs());
        put_limbs(&mut chunk[32..64], b.inner.y.to_montgomery_limbs());
    }
    let mut out = [0u8; 128];
    check(unsafe {
        d377_msm(ws.as_ptr(), wp.as_ptr(), PT_AFFINE | SCALARS_MONTGOMERY, n, out.as_mut_ptr(), core::ptr::null_mut())
    })?;
    Ok(wire_to_element(&out))
}

/// Long-lived MSM bases on the GPU: `ScalarMul::batch_convert_to_mul_base` once
/// (ark_curve/element.rs:27-34), `VariableBaseMSM::msm(&bases, &scalars)` many times
/// (element.rs:37).  Only the 32-byte scalars cross the link per call.
pub struct GpuBases {
    ptr: *mut u8,
    len: usize,
}

// The handle is an opaque device pointer; the library serialises calls per engine.
unsafe impl Send for GpuBases {}

impl GpuBases {
    pub fn new(points: &[Element]) -> Result<Self, GpuError> {
        let w = elements_to_wire(points);
        let mut ptr: *mut u8 = core::ptr::null_mut();
        check(unsafe { d377_msm_bases_create(w.as_ptr(), PT_ELEMENT, points.len(), &mut ptr) })?;
        Ok(GpuBases { ptr, len: points.len() })
    }

    /// The same bases with the window multiples 2^(c j) * P_i precomputed
    /// (d377_msm_bases_create_windowed: n * ceil(252 / c) * 128 bytes of device memory, and
    /// every `msm` skips the Horner tail).  `c` = 0 lets the library choose from n.
    pub fn new_windowed(points: &[Element], c: i32) -> Result<Self, GpuError> {
        let w = elements_to_wire(points);
        let mut ptr: *mut u8 = core::ptr::null_mut();
        check(unsafe { d377_msm_bases_create_windowed(w.as_ptr(), PT_ELEMENT, points.len(), c as c_int, &mut ptr) })?;
        Ok(GpuBases { ptr, len: points.len() })
    }

    /// (window width c, windows W, device bytes) of the set: (0, 1, _) for `new`.
    pub fn layout(&self) -> Result<(i32, i32, usize), GpuError> {
        let (mut n, mut c, mut w, mut bytes) = (0usize, 0 as c_int, 0 as c_int, 0usize);
        check(unsafe { d377_msm_bases_info(self.ptr as *const u8, &mut n, &mut c, &mut w, &mut bytes) })?;
        Ok((c as i32, w as i32, bytes))
    }

    pub fn len(&self) -> usize {
        self.len
    }

    pub fn is_empty(&self) -> bool {
        self.len == 0
    }

    /// MSM over the first `scalars.len()` bases (at most `self.len()` scalars are used).
    pub fn msm(&self, scalars: &[Fr]) -> Result<Element, GpuError> {
        let n = core::cmp::min(scalars.len(), self.len);
        let ws = scalars_to_wire(&scalars[..n]);
        let mut out = [0u8; 128];
        check(unsafe {
            d377_msm(ws.as_ptr(), self.ptr as *const u8, PT_BASES | SCALARS_MONTGOMERY, n, out.as_mut_ptr(),
                     core::ptr::null_mut())
        })?;
        Ok(wire_to_element(&out))
    }
}

impl Drop for GpuBases {
    fn drop(&mut self) {
        if !self.ptr.is_null() {
            // after d377_shutdown the library has released the bases itself and reports
            // NOT_INITIALISED here; there is nothing left to free either way
            let _ = unsafe { d377_msm_bases_destroy(self.ptr) };
            self.ptr = core::ptr::null_mut();
        }
    }
}

/// Fixed-base window tables of k long-lived points B_0..B_{k-1} (d377_fixed_bases_create:
/// 48 MiB of device memory per base).  `mul` computes `sum_j s_ij * B_j` for every row i of
/// k scalars -- with k = 1 `B * s` for many s, with k = 2 e.g. Pedersen commitments
/// `v * G_a + r * H` -- at 16 k mixed additions per row instead of k variable-base ladders.
pub struct GpuFixedBases {
    ptr: *mut u8,
    len: usize,
}

// The handle is an opaque device pointer; the library serialises calls per engine.
unsafe impl Send for GpuFixedBases {}

impl GpuFixedBases {
    pub fn new(points: &[Element]) -> Result<Self, GpuError> {
        let w = elements_to_wire(points);
        let mut ptr: *mut u8 = core::ptr::null_mut();
        check(unsafe { d377_fixed_bases_create(w.as_ptr(), PT_ELEMENT, points.len(), &mut ptr) })?;
        Ok(GpuFixedBases { ptr, len: points.len() })
    }

    /// k, the number of bases (and of scalars per row).
    pub fn len(&self) -> usize {
        self.len
    }

    pub fn is_empty(&self) -> bool {
        self.len == 0
    }

    fn run(&self, scalars: &[Fr], out_format: c_int, width: usize) -> Result<Vec<u8>, GpuError> {
        assert!(scalars.len() % self.len == 0, "scalars: rows of k = {} scalars", self.len);
        let n = scalars.len() / self.len;
        let ws = scalars_to_wire(scalars);
        let mut out = vec![0u8; width * n];
        check(unsafe {
            d377_fixed_bases_mul(self.ptr as *const u8, ws.as_ptr(), n, out.as_mut_ptr(), out_format | SCALARS_MONTGOMERY)
        })?;
        Ok(out)
    }

    /// `sum_j scalars[i * k + j] * B_j` for every row i; `scalars` is row-major, its length a
    /// multiple of k.
    pub fn mul(&self, scalars: &[Fr]) -> Result<Vec<Element>, GpuError> {
        Ok(wire_to_elements(&self.run(scalars, OUT_ELEMENT, 128)?))
    }

    /// The same, `vartime_compress`ed in the same launch.
    pub fn mul_compressed(&self, scalars: &[Fr]) -> Result<Vec<Encoding>, GpuError> {
        Ok(wire_to_encodings(&self.run(scalars, OUT_ENCODING, 32)?))
    }
}

impl Drop for GpuFixedBases {
    fn drop(&mut self) {
        if !self.ptr.is_null() {
            // after d377_shutdown the library has released the tables itself
            let _ = unsafe { d377_fixed_bases_destroy(self.ptr) };
            self.ptr = core::ptr::null_mut();
        }
    }
}

/// Page-locked staging buffer (`d377_host_alloc`): callers that build the wire images
/// themselves (e.g. a prover that keeps its scalars in one allocation) get full PCIe speed
/// and overlapped upload / compute from the host-buffer entry points with it.
pub struct PinnedBuf {
    ptr: *mut u8,
    len: usize,
}

unsafe impl Send for PinnedBuf {}

impl PinnedBuf {
    pub fn new(len: usize) -> Result<Self, GpuError> {
        let p = unsafe { d377_host_alloc(len) } as *mut u8;
        if p.is_null() {
            return Err(GpuError { code: D377_ERR_CUDA, message: "d377_host_alloc failed".into() });
        }
        Ok(PinnedBuf { ptr: p, len })
    }

    pub fn as_mut_slice(&mut self) -> &mut [u8] {
        // SAFETY: `ptr` is a live allocation of `len` bytes owned by this value.
        unsafe { core::slice::from_raw_parts_mut(self.ptr, self.len) }
    }

    pub fn as_slice(&self) -> &[u8] {
        unsafe { core::slice::from_raw_parts(self.ptr, self.len) }
    }
}

impl Drop for PinnedBuf {
    fn drop(&mut self) {
        let _ = unsafe { d377_host_free(self.ptr as *mut c_void) };
    }
}

// ---------------------------------------------------------------------------------------------
// tests (cargo test --features b200 on a box with a B200): the crate's own properties,
// batch against per-element
// ---------------------------------------------------------------------------------------------
#[cfg(test)]
mod tests {
    use super::*;

    fn points(n: usize) -> Vec<Element> {
        // tests/operations.rs:6-11
        (0..n as u64).map(|i| Element::encode_to_curve(&Fq::from(i + 1))).collect()
    }

    fn scalars(n: usize) -> Vec<Fr> {
        (0..n as u64).map(|i| Fr::from(i * i + 7) * Fr::from(0x9e37_79b9_7f4a_7c15u64)).collect()
    }

    #[test]
    fn batch_matches_per_element() {
        init(0).unwrap();
        let p = points(257);
        let s = scalars(257);
        let enc = compress_batch(&p).unwrap();
        for (e, q) in enc.iter().zip(p.iter()) {
            assert_eq!(*e, q.vartime_compress());
        }
        let back = decompress_batch(&enc).unwrap();
        for (b, q) in back.iter().zip(p.iter()) {
            assert_eq!(b.as_ref().unwrap(), q);
        }
        let prod = mul_batch(&p, &s).unwrap();
        for i in 0..p.len() {
            assert_eq!(prod[i], p[i] * s[i]);
        }
        // tests/operations.rs:44-60
        let msm = vartime_multiscalar_mul(&s, &p).unwrap();
        assert_eq!(msm, Element::vartime_multiscalar_mul(s.iter(), p.iter()));
        let bases = GpuBases::new(&p).unwrap();
        assert_eq!(bases.msm(&s).unwrap(), msm);
        let win = GpuBases::new_windowed(&p, 0).unwrap();
        assert_eq!(win.msm(&s).unwrap(), msm);
        // k = 2 fixed bases: rows (s_i, s_{i+1}) against (p_0, p_1)
        let fb = GpuFixedBases::new(&p[..2]).unwrap();
        assert_eq!(fb.len(), 2);
        let lc = fb.mul(&s[..16]).unwrap();
        let lc_enc = fb.mul_compressed(&s[..16]).unwrap();
        for i in 0..8 {
            let want = p[0] * s[2 * i] + p[1] * s[2 * i + 1];
            assert_eq!(lc[i], want);
            assert_eq!(lc_enc[i], want.vartime_compress());
        }
        let g = generator_mul_batch(&s).unwrap();
        for i in 0..s.len() {
            assert_eq!(g[i], Element::GENERATOR * s[i]);
        }
        assert!(is_on_curve_batch(&p, true).unwrap().into_iter().all(|b| b));
        // ark_curve/serialize.rs:8-46: the AffinePoint wire format, both directions
        let aff = normalize_batch(&p).unwrap();
        let ser = serialize_affine_batch(&aff).unwrap();
        assert_eq!(ser, enc);
        let de = deserialize_affine_batch(&ser).unwrap();
        for (a, e) in de.iter().zip(enc.iter()) {
            let mut bytes = Vec::new();
            ark_serialize::CanonicalSerialize::serialize_compressed(a.as_ref().unwrap(), &mut bytes).unwrap();
            assert_eq!(&bytes[..], &e.0[..]);
        }
    }

    #[test]
    fn invalid_encodings_are_per_element_errors() {
        init(0).unwrap();
        let mut bad = [0u8; 32];
        bad[0] = 1; // tests/encoding.rs:28-52
        let r = decompress_batch(&[Encoding([0u8; 32]), Encoding(bad)]).unwrap();
        assert!(r[0].as_ref().unwrap().is_identity());
        assert!(matches!(r[1], Err(EncodingError::InvalidEncoding)));
        let a = deserialize_affine_batch(&[Encoding([0u8; 32]), Encoding(bad)]).unwrap();
        assert!(a[0].is_ok());
        assert!(matches!(a[1], Err(EncodingError::InvalidEncoding)));
    }
}
