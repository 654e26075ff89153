//! babyjubjub-rs API over the B200 batch engine (libbjj_cuda).
//!
//! UNTESTED SOURCE: the build image has no Rust toolchain.  The same C ABI is exercised by the Python
//! (`babyjubjub-rs_b200/`) and C++ (`host/bjj.hpp`) mirrors, which the parity tests drive.
//!
//! The public names follow arnaucube/babyjubjub-rs 0.0.11: `Point`, `PointProjective`, `Signature`,
//! `PrivateKey`, `decompress_point`, `decompress_signature`, `verify`, plus the batch entry points
//! `mul_scalar_batch`, `public_batch`, `decompress_batch`, `verify_batch`, and `FixedBase` (k*P and k*P + l*Q on
//! the comb table of a caller-chosen point).  `Fr` is carried as its
//! canonical 32-byte little-endian value (what ff_ce's `into_repr()` yields).  There is no CPU
//! fallback: without a CUDA device `Engine::new` returns an error.
pub mod ffi;

use num_bigint::{BigInt, Sign};
use std::ffi::CStr;
use std::sync::{Mutex, MutexGuard, OnceLock};

/// The reference's `Fr` is `poseidon_rs::Fr` (an ff_ce field element, src/lib.rs:7).  This crate has no field
/// arithmetic on the host -- every operation runs on the device -- so a field element is carried as the canonical
/// 32 little-endian bytes that `into_repr()` yields.  A maintainer who keeps `poseidon_rs::Fr` in the public types
/// converts at this boundary with `fr_to_le32` / `fr_from_le32` (INTEGRATION.md).
pub type Fr = [u8; 32];

pub fn q() -> BigInt {
    BigInt::parse_bytes(b"21888242871839275222246405745257275088548364400416034343698204186575808495617", 10).unwrap()
}

pub fn fr_from_str(s: &str) -> Option<Fr> {
    let v = BigInt::parse_bytes(s.as_bytes(), 10)?;
    if v.sign() == Sign::Minus {
        return None;
    }
    Some(bigint_le32(&(v % q())))
}

pub fn suborder() -> BigInt {
    BigInt::parse_bytes(b"2736030358979909402780800718157159386076813972158567259200215660948447373041", 10).unwrap()
}

/// 32 little-endian bytes of |v|.  Panics if |v| needs more than 256 bits: callers that may hold wider values go
/// through `scalar_b8_le32` (scalars of B8) or the wide entry point (`mul_scalar_batch`).
pub fn bigint_le32(v: &BigInt) -> [u8; 32] {
    let (_, bytes) = v.to_bytes_le();
    assert!(bytes.len() <= 32, "value wider than 256 bits");
    let mut out = [0u8; 32];
    out[..bytes.len()].copy_from_slice(&bytes);
    out
}

/// A scalar that multiplies B8 (S of `verify`, s of `verify_schnorr`, k of `sign_schnorr`).  The reference hands the
/// BigInt to `B8.mul_scalar` as it is (sign dropped, src/lib.rs:156); B8 has order SUBORDER, so a value wider than
/// 256 bits is reduced mod SUBORDER -- the same group element.  Narrower values cross the ABI unreduced.
pub fn scalar_b8_le32(v: &BigInt) -> [u8; 32] {
    let m = v.magnitude();
    if m.bits() <= 256 {
        bigint_le32(v)
    } else {
        bigint_le32(&(BigInt::from(m.clone()) % suborder()))
    }
}

fn msg_le32(msg: &BigInt) -> [u8; 32] {
    // `verify` returns false for msg > Q; any 32-byte value > Q carries that through the ABI
    if msg > &q() {
        [0xFF; 32]
    } else {
        bigint_le32(msg)
    }
}

/// One `bjj_ctx` on one device.  The C context is NOT thread-safe (one host thread at a time: it owns streams,
/// staging arenas and scratch), while the reference's free functions are; so the context may move between threads
/// (`Send`) but is never shared (`!Sync`), and the process-wide engine below sits behind a `Mutex` that every FFI
/// call takes.  For parallel callers use one `Engine` per thread, or `MultiEngine` for one batch over all devices.
pub struct Engine {
    ctx: *mut ffi::bjj_ctx,
}
unsafe impl Send for Engine {}

impl Engine {
    pub fn new(device: i32) -> Result<Engine, String> {
        let mut ctx = std::ptr::null_mut();
        let rc = unsafe { ffi::bjj_init(device, &mut ctx) };
        if rc != ffi::BJJ_OK {
            return Err(format!("bjj_init failed: {} (there is no CPU fallback)", err_str(rc)));
        }
        Ok(Engine { ctx })
    }
    pub fn raw(&self) -> *mut ffi::bjj_ctx {
        self.ctx
    }
}
impl Drop for Engine {
    fn drop(&mut self) {
        unsafe { ffi::bjj_destroy(self.ctx) }
    }
}

fn err_str(rc: i32) -> String {
    unsafe { CStr::from_ptr(ffi::bjj_error_string(rc)).to_string_lossy().into_owned() }
}
fn status_str(st: u8) -> String {
    unsafe { CStr::from_ptr(ffi::bjj_status_string(st as i32)).to_string_lossy().into_owned() }
}
fn check(rc: i32, what: &str) {
    assert!(rc == ffi::BJJ_OK, "{} failed: {}", what, err_str(rc));
}

static ENGINE: OnceLock<Mutex<Engine>> = OnceLock::new();
/// The process-wide engine (device 0), locked for the duration of the caller's FFI call.
pub fn engine() -> MutexGuard<'static, Engine> {
    ENGINE
        .get_or_init(|| Mutex::new(Engine::new(0).expect("CUDA device required")))
        .lock()
        .unwrap_or_else(|e| e.into_inner())
}

fn col<F: Fn(usize) -> [u8; 32]>(n: usize, f: F) -> Vec<u8> {
    let mut v = Vec::with_capacity(32 * n);
    for i in 0..n {
        v.extend_from_slice(&f(i));
    }
    v
}
fn row(buf: &[u8], i: usize) -> [u8; 32] {
    let mut r = [0u8; 32];
    r.copy_from_slice(&buf[32 * i..32 * i + 32]);
    r
}

#[derive(Clone, Debug, PartialEq)]
pub struct PointProjective {
    pub x: Fr,
    pub y: Fr,
    pub z: Fr,
}

#[derive(Clone, Debug, PartialEq)]
pub struct Point {
    pub x: Fr,
    pub y: Fr,
}

impl PointProjective {
    pub fn affine(&self) -> Point {
        let (mut rx, mut ry) = ([0u8; 32], [0u8; 32]);
        check(unsafe { ffi::bjj_affine_batch(engine().raw(), 1, self.x.as_ptr(), self.y.as_ptr(), self.z.as_ptr(),
                                             rx.as_mut_ptr(), ry.as_mut_ptr()) }, "bjj_affine_batch");
        Point { x: rx, y: ry }
    }
    pub fn add(&self, q: &PointProjective) -> PointProjective {
        let (mut rx, mut ry, mut rz) = ([0u8; 32], [0u8; 32], [0u8; 32]);
        check(unsafe { ffi::bjj_add_batch(engine().raw(), 1, self.x.as_ptr(), self.y.as_ptr(), self.z.as_ptr(),
                                          q.x.as_ptr(), q.y.as_ptr(), q.z.as_ptr(), rx.as_mut_ptr(), ry.as_mut_ptr(),
                                          rz.as_mut_ptr()) }, "bjj_add_batch");
        PointProjective { x: rx, y: ry, z: rz }
    }
}

impl Point {
    pub fn projective(&self) -> PointProjective {
        let mut one = [0u8; 32];
        one[0] = 1;
        PointProjective { x: self.x, y: self.y, z: one }
    }
    pub fn mul_scalar(&self, n: &BigInt) -> Point {
        mul_scalar_batch(std::slice::from_ref(self), std::slice::from_ref(n)).pop().unwrap()
    }
    pub fn compress(&self) -> [u8; 32] {
        let mut out = [0u8; 32];
        check(unsafe { ffi::bjj_compress_batch(engine().raw(), 1, self.x.as_ptr(), self.y.as_ptr(), out.as_mut_ptr()) },
              "bjj_compress_batch");
        out
    }
    pub fn equals(&self, p: Point) -> bool {
        self.x == p.x && self.y == p.y
    }
}

pub fn decompress_point(bb: [u8; 32]) -> Result<Point, String> {
    decompress_batch(&[bb]).pop().unwrap()
}

#[derive(Debug, Clone)]
pub struct Signature {
    pub r_b8: Point,
    pub s: BigInt,
}
impl Signature {
    pub fn compress(&self) -> [u8; 64] {
        let mut r = [0u8; 64];
        r[..32].copy_from_slice(&self.r_b8.compress());
        // src/lib.rs:250-254: the low 32 little-endian bytes of S (signatures made by `sign` have S < SUBORDER)
        let (_, sb) = self.s.to_bytes_le();
        let m = sb.len().min(32);
        r[32..32 + m].copy_from_slice(&sb[..m]);
        r
    }
}
pub fn decompress_signature(b: &[u8; 64]) -> Result<Signature, String> {
    let mut rb = [0u8; 32];
    rb.copy_from_slice(&b[..32]);
    let r_b8 = decompress_point(rb)?;
    Ok(Signature { r_b8, s: BigInt::from_bytes_le(Sign::Plus, &b[32..]) })
}

pub struct PrivateKey {
    pub key: [u8; 32],
}
impl PrivateKey {
    pub fn import(b: Vec<u8>) -> Result<PrivateKey, String> {
        if b.len() != 32 {
            return Err(String::from("imported key can not be bigger than 32 bytes"));
        }
        let mut key = [0u8; 32];
        key.copy_from_slice(&b);
        Ok(PrivateKey { key })
    }
    pub fn scalar_key(&self) -> BigInt {
        let mut out = [0u8; 32];
        check(unsafe { ffi::bjj_scalar_key_batch(engine().raw(), 1, self.key.as_ptr(), out.as_mut_ptr()) },
              "bjj_scalar_key_batch");
        BigInt::from_bytes_le(Sign::Plus, &out)
    }
    pub fn public(&self) -> Point {
        public_batch(std::slice::from_ref(self)).pop().unwrap()
    }
    pub fn sign(&self, msg: BigInt) -> Result<Signature, String> {
        if msg > q() {
            return Err("msg outside the Finite Field".to_string());
        }
        let m = bigint_le32(&msg);
        let (mut rx, mut ry, mut s, mut st) = ([0u8; 32], [0u8; 32], [0u8; 32], 0u8);
        check(unsafe { ffi::bjj_sign_batch(engine().raw(), 1, self.key.as_ptr(), m.as_ptr(), rx.as_mut_ptr(),
                                           ry.as_mut_ptr(), s.as_mut_ptr(), &mut st) }, "bjj_sign_batch");
        if st != 0 {
            return Err(status_str(st));
        }
        Ok(Signature { r_b8: Point { x: rx, y: ry }, s: BigInt::from_bytes_le(Sign::Plus, &s) })
    }
}

impl PrivateKey {
    /// src/lib.rs:345-362.  `k` is the caller's nonce (the reference draws 1024 random bits from `rand`; this crate
    /// has no RNG dependency): r = B8*k, h = schnorr_hash(pk, m, r), s = k + scalar_key*h, unreduced like the reference.
    pub fn sign_schnorr_with_nonce(&self, m: BigInt, k: &BigInt) -> Result<(Point, BigInt), String> {
        let kb = scalar_b8_le32(k);
        let (mut rx, mut ry) = ([0u8; 32], [0u8; 32]);
        check(unsafe { ffi::bjj_fixed_base_batch(engine().raw(), 1, kb.as_ptr(), rx.as_mut_ptr(), ry.as_mut_ptr()) },
              "bjj_fixed_base_batch");
        let r = Point { x: rx, y: ry };
        let h = schnorr_hash(&self.public(), m, &r)?;
        Ok((r, k + &self.scalar_key() * &h))
    }
}

/// src/lib.rs:364-373
pub fn schnorr_hash(pk: &Point, msg: BigInt, c: &Point) -> Result<BigInt, String> {
    if msg > q() {
        return Err("msg outside the Finite Field".to_string());
    }
    let m = bigint_le32(&(msg % q()));
    let ins: [*const u8; 5] = [pk.x.as_ptr(), pk.y.as_ptr(), c.x.as_ptr(), c.y.as_ptr(), m.as_ptr()];
    let mut out = [0u8; 32];
    check(unsafe { ffi::bjj_poseidon_batch(engine().raw(), 5, 1, ins.as_ptr(), out.as_mut_ptr()) }, "bjj_poseidon_batch");
    Ok(BigInt::from_bytes_le(Sign::Plus, &out))
}

/// src/lib.rs:375-385: s*B8 == r + h*pk
pub fn verify_schnorr(pk: Point, m: BigInt, r: Point, s: BigInt) -> Result<bool, String> {
    let mb = msg_le32(&m);
    let sb = scalar_b8_le32(&s);
    let (mut ok, mut st) = (0u8, 0u8);
    check(unsafe { ffi::bjj_verify_schnorr_batch(engine().raw(), 1, pk.x.as_ptr(), pk.y.as_ptr(), mb.as_ptr(), r.x.as_ptr(),
                                                 r.y.as_ptr(), sb.as_ptr(), &mut ok, &mut st) }, "bjj_verify_schnorr_batch");
    if st != 0 {
        return Err(status_str(st));
    }
    Ok(ok == 1)
}

/// Inputs of the verify_schnorr batches: messages and `(r, s)` pairs as `sign_schnorr_batch_with_nonces` returns them,
/// s (sign dropped) in the smallest multiple of 256 bits that holds the widest.  Panics on a negative msg, on s wider than
/// 2304 bits, or on lengths that differ.
struct SchnorrLanes {
    n: usize,
    words: usize,
    m: Vec<u8>,
    rx: Vec<u8>,
    ry: Vec<u8>,
    s: Vec<u8>,
}
fn schnorr_lanes(msgs: &[BigInt], sigs: &[(Point, BigInt)]) -> SchnorrLanes {
    let n = sigs.len();
    assert_eq!(n, msgs.len());
    assert!(msgs.iter().all(|m| m.sign() != Sign::Minus), "negative msg");
    let bits = sigs.iter().map(|(_, s)| s.bits()).max().unwrap_or(0).max(1);
    assert!(bits <= 2304, "s wider than 2304 bits");
    let words = (8 * ((bits + 255) / 256)) as usize;
    let mut s = vec![0u8; 4 * words * n];
    for (i, (_, v)) in sigs.iter().enumerate() {
        let (_, bytes) = v.to_bytes_le();
        s[4 * words * i..4 * words * i + bytes.len()].copy_from_slice(&bytes);
    }
    SchnorrLanes { n, words, m: col(n, |i| msg_le32(&msgs[i])), rx: col(n, |i| sigs[i].0.x), ry: col(n, |i| sigs[i].0.y), s }
}
fn schnorr_results(ok: &[u8], st: &[u8]) -> Vec<Result<bool, String>> {
    (0..ok.len()).map(|i| if st[i] == 0 { Ok(ok[i] == 1) } else { Err(status_str(st[i])) }).collect()
}

/// `verify_schnorr(pks[i], msgs[i], r, s)` (src/lib.rs:364-385) lane by lane on the signer's unreduced `(r, s)`, reduced
/// mod SUBORDER on the device
pub fn verify_schnorr_batch(pks: &[Point], msgs: &[BigInt], sigs: &[(Point, BigInt)]) -> Vec<Result<bool, String>> {
    let l = schnorr_lanes(msgs, sigs);
    assert_eq!(l.n, pks.len());
    let (ax, ay) = (col(l.n, |i| pks[i].x), col(l.n, |i| pks[i].y));
    let (mut ok, mut st) = (vec![0u8; l.n], vec![0u8; l.n]);
    check(unsafe { ffi::bjj_verify_schnorr_wide_batch(engine().raw(), l.n, ax.as_ptr(), ay.as_ptr(), l.m.as_ptr(), l.rx.as_ptr(),
                                                      l.ry.as_ptr(), l.s.as_ptr(), l.words as i32, ok.as_mut_ptr(),
                                                      st.as_mut_ptr()) }, "bjj_verify_schnorr_wide_batch");
    schnorr_results(&ok, &st)
}

/// src/lib.rs:387-393 draws 1024 random bits and keeps the first 32 big-endian bytes; here the caller supplies the
/// 32 random bytes (no RNG dependency in this crate).
pub fn new_key_from_bytes(random32: [u8; 32]) -> PrivateKey {
    PrivateKey { key: random32 }
}

pub fn verify(pk: Point, sig: Signature, msg: BigInt) -> bool {
    verify_batch(&[pk], &[sig], &[msg])[0]
}

// ---- batch entry points ------------------------------------------------------------------------------

/// `Point::mul_scalar` over a batch (src/lib.rs:149-164).  Scalars are BigInts of any size up to 2048 bits, sign
/// dropped as in the reference (:156).  Up to 256 bits they cross the ABI as they are; wider batches use
/// `bjj_mul_scalar_wide_batch` (on-curve points: reduced mod ORDER on the device, exact; off-curve points: every bit
/// of the wide scalar is replayed like the reference's loop).
pub fn mul_scalar_batch(points: &[Point], scalars: &[BigInt]) -> Vec<Point> {
    let n = points.len();
    assert_eq!(n, scalars.len());
    let (px, py) = (col(n, |i| points[i].x), col(n, |i| points[i].y));
    let (mut rx, mut ry) = (vec![0u8; 32 * n], vec![0u8; 32 * n]);
    let bits = scalars.iter().map(|k| k.bits()).max().unwrap_or(0);
    if bits <= 256 {
        let k = col(n, |i| bigint_le32(&scalars[i]));
        check(unsafe { ffi::bjj_mul_scalar_batch(engine().raw(), n, px.as_ptr(), py.as_ptr(), k.as_ptr(), rx.as_mut_ptr(),
                                                 ry.as_mut_ptr()) }, "bjj_mul_scalar_batch");
    } else {
        let words = 8 * ((bits as usize + 255) / 256);
        assert!(words <= 64, "scalars wider than 2048 bits are not supported by the device ABI");
        let mut k = vec![0u8; 4 * words * n];
        for i in 0..n {
            let (_, b) = scalars[i].to_bytes_le();
            k[4 * words * i..4 * words * i + b.len()].copy_from_slice(&b);
        }
        check(unsafe { ffi::bjj_mul_scalar_wide_batch(engine().raw(), n, px.as_ptr(), py.as_ptr(), k.as_ptr(), words as i32,
                                                      rx.as_mut_ptr(), ry.as_mut_ptr()) }, "bjj_mul_scalar_wide_batch");
    }
    (0..n).map(|i| Point { x: row(&rx, i), y: row(&ry, i) }).collect()
}

/// Reduces a scalar for the fixed-base tables: the reference multiplies by |k| (sign dropped, src/lib.rs:156); every
/// on-curve point has an order dividing ORDER, so a |k| wider than 256 bits is reduced mod ORDER -- the same point.
pub fn scalar_base_le32(v: &BigInt) -> [u8; 32] {
    let m = v.magnitude();
    if m.bits() <= 256 {
        bigint_le32(v)
    } else {
        bigint_le32(&(BigInt::from(m.clone()) % (suborder() * 8)))
    }
}

/// The comb table of one on-curve point P (50 MB of device memory on the process-wide engine's device, freed on drop):
/// `P.mul_scalar(k)` for many `k` at the rate of B8's fixed-base path, and `k*P + l*Q` in one pass.  An off-curve P has
/// no table (its reference result depends on mul_scalar's exact double-and-add order): `new` returns Err and the caller
/// keeps `mul_scalar_batch`.
pub struct FixedBase {
    base: *mut ffi::bjj_base,
}
unsafe impl Send for FixedBase {}

impl FixedBase {
    pub fn new(p: &Point) -> Result<FixedBase, String> {
        let mut base = std::ptr::null_mut();
        let rc = unsafe { ffi::bjj_base_create(engine().raw(), p.x.as_ptr(), p.y.as_ptr(), &mut base) };
        if rc != ffi::BJJ_OK {
            return Err(format!("bjj_base_create failed: {}", err_str(rc)));
        }
        Ok(FixedBase { base })
    }
    /// `[P.mul_scalar(k) for k in scalars]`
    pub fn mul_batch(&self, scalars: &[BigInt]) -> Vec<Point> {
        let n = scalars.len();
        let k = col(n, |i| scalar_base_le32(&scalars[i]));
        let (mut rx, mut ry) = (vec![0u8; 32 * n], vec![0u8; 32 * n]);
        check(unsafe { ffi::bjj_base_mul_batch(engine().raw(), self.base, n, k.as_ptr(), rx.as_mut_ptr(), ry.as_mut_ptr()) },
              "bjj_base_mul_batch");
        (0..n).map(|i| Point { x: row(&rx, i), y: row(&ry, i) }).collect()
    }
    /// `(k*P).projective().add((l*Q).projective()).affine()` lane by lane; `q == None` selects B8
    pub fn mul2_batch(&self, ks: &[BigInt], q: Option<&FixedBase>, ls: &[BigInt]) -> Vec<Point> {
        let n = ks.len();
        assert_eq!(n, ls.len());
        let (k, l) = (col(n, |i| scalar_base_le32(&ks[i])), col(n, |i| scalar_base_le32(&ls[i])));
        let qb = q.map_or(std::ptr::null(), |b| b.base as *const ffi::bjj_base);
        let (mut rx, mut ry) = (vec![0u8; 32 * n], vec![0u8; 32 * n]);
        check(unsafe { ffi::bjj_base_mul2_batch(engine().raw(), self.base, qb, n, k.as_ptr(), l.as_ptr(), rx.as_mut_ptr(),
                                                ry.as_mut_ptr()) }, "bjj_base_mul2_batch");
        (0..n).map(|i| Point { x: row(&rx, i), y: row(&ry, i) }).collect()
    }
    /// `verify(P, sig, msg)` (src/lib.rs:395-412) lane by lane for signatures of the one key P: the results of
    /// `verify_batch` with P in every lane, from the two comb tables
    pub fn verify_batch(&self, sigs: &[Signature], msgs: &[BigInt]) -> Vec<bool> {
        let n = sigs.len();
        assert_eq!(n, msgs.len());
        let (r8x, r8y) = (col(n, |i| sigs[i].r_b8.x), col(n, |i| sigs[i].r_b8.y));
        let s = col(n, |i| scalar_b8_le32(&sigs[i].s));
        let m = col(n, |i| msg_le32(&msgs[i]));
        let mut ok = vec![0u8; n];
        check(unsafe { ffi::bjj_verify_base_batch(engine().raw(), self.base, n, r8x.as_ptr(), r8y.as_ptr(), s.as_ptr(),
                                                  m.as_ptr(), ok.as_mut_ptr()) }, "bjj_verify_base_batch");
        ok.into_iter().map(|b| b == 1).collect()
    }
    /// the same from 64-byte compressed signatures: `Err` carries R8's decompression error
    pub fn verify_compressed_batch(&self, sigs: &[[u8; 64]], msgs: &[BigInt]) -> Vec<Result<bool, String>> {
        let n = sigs.len();
        assert_eq!(n, msgs.len());
        let sg: Vec<u8> = sigs.iter().flat_map(|s| s.iter().copied()).collect();
        let m = col(n, |i| msg_le32(&msgs[i]));
        let (mut ok, mut st) = (vec![0u8; n], vec![0u8; n]);
        check(unsafe { ffi::bjj_verify_base_compressed_batch(engine().raw(), self.base, n, sg.as_ptr(), m.as_ptr(),
                                                             ok.as_mut_ptr(), st.as_mut_ptr()) },
              "bjj_verify_base_compressed_batch");
        (0..n).map(|i| if st[i] == 0 { Ok(ok[i] == 1) } else { Err(status_str(st[i])) }).collect()
    }
    /// `verify_schnorr_batch` with P in every lane, on the comb tables
    pub fn verify_schnorr_batch(&self, msgs: &[BigInt], sigs: &[(Point, BigInt)]) -> Vec<Result<bool, String>> {
        let l = schnorr_lanes(msgs, sigs);
        let (mut ok, mut st) = (vec![0u8; l.n], vec![0u8; l.n]);
        check(unsafe { ffi::bjj_verify_schnorr_base_batch(engine().raw(), self.base, l.n, l.m.as_ptr(), l.rx.as_ptr(), l.ry.as_ptr(),
                                                          l.s.as_ptr(), l.words as i32, ok.as_mut_ptr(), st.as_mut_ptr()) },
              "bjj_verify_schnorr_base_batch");
        schnorr_results(&ok, &st)
    }
}
impl Drop for FixedBase {
    fn drop(&mut self) {
        unsafe { ffi::bjj_base_destroy(engine().raw(), self.base) }
    }
}

/// N on-curve public keys with compact comb tables (396,480 B of device memory per key): verify and k*P for batches
/// that name a key per lane.  Freed on drop.
pub struct KeySet {
    ks: *mut ffi::bjj_keyset,
}
unsafe impl Send for KeySet {}

impl KeySet {
    /// `Err` for an empty list, a coordinate >= Q or an off-curve key; `key_status` says which keys and why
    pub fn new(keys: &[Point]) -> Result<KeySet, (String, Vec<u8>)> {
        let n = keys.len();
        let (ax, ay) = (col(n, |i| keys[i].x), col(n, |i| keys[i].y));
        let mut st = vec![0u8; n];
        let mut ks = std::ptr::null_mut();
        let rc = unsafe { ffi::bjj_keyset_create(engine().raw(), n, ax.as_ptr(), ay.as_ptr(), st.as_mut_ptr(), &mut ks) };
        if rc != ffi::BJJ_OK {
            return Err((format!("bjj_keyset_create failed: {}", err_str(rc)), st));
        }
        Ok(KeySet { ks })
    }
    /// adds keys under the indices after the last; existing indices keep their keys.  `Err` as for `new`, and the set
    /// is then unchanged
    pub fn append(&mut self, keys: &[Point]) -> Result<(), (String, Vec<u8>)> {
        let n = keys.len();
        let (ax, ay) = (col(n, |i| keys[i].x), col(n, |i| keys[i].y));
        let mut st = vec![0u8; n];
        let rc = unsafe { ffi::bjj_keyset_append(engine().raw(), self.ks, n, ax.as_ptr(), ay.as_ptr(), st.as_mut_ptr()) };
        if rc != ffi::BJJ_OK {
            return Err((format!("bjj_keyset_append failed: {}", err_str(rc)), st));
        }
        Ok(())
    }
    /// gives keys `first ..` new coordinates (key rotation).  `Err` as for `new` or for a range past the set, and the
    /// set is then unchanged
    pub fn replace(&mut self, first: usize, keys: &[Point]) -> Result<(), (String, Vec<u8>)> {
        let n = keys.len();
        let (ax, ay) = (col(n, |i| keys[i].x), col(n, |i| keys[i].y));
        let mut st = vec![0u8; n];
        let rc = unsafe { ffi::bjj_keyset_replace(engine().raw(), self.ks, first, n, ax.as_ptr(), ay.as_ptr(), st.as_mut_ptr()) };
        if rc != ffi::BJJ_OK {
            return Err((format!("bjj_keyset_replace failed: {}", err_str(rc)), st));
        }
        Ok(())
    }
    /// `verify(keys[key_index[i]], sigs[i], msgs[i])` (src/lib.rs:395-412) lane by lane: the results of `verify_batch`
    /// with those keys
    pub fn verify_batch(&self, key_index: &[u32], sigs: &[Signature], msgs: &[BigInt]) -> Vec<bool> {
        let n = sigs.len();
        assert_eq!(n, msgs.len());
        assert_eq!(n, key_index.len());
        let (r8x, r8y) = (col(n, |i| sigs[i].r_b8.x), col(n, |i| sigs[i].r_b8.y));
        let s = col(n, |i| scalar_b8_le32(&sigs[i].s));
        let m = col(n, |i| msg_le32(&msgs[i]));
        let mut ok = vec![0u8; n];
        check(unsafe { ffi::bjj_verify_keyset_batch(engine().raw(), self.ks, n, key_index.as_ptr(), r8x.as_ptr(), r8y.as_ptr(),
                                                    s.as_ptr(), m.as_ptr(), ok.as_mut_ptr()) }, "bjj_verify_keyset_batch");
        ok.into_iter().map(|b| b == 1).collect()
    }
    /// the same from 64-byte compressed signatures: `Err` carries R8's decompression error
    pub fn verify_compressed_batch(&self, key_index: &[u32], sigs: &[[u8; 64]], msgs: &[BigInt]) -> Vec<Result<bool, String>> {
        let n = sigs.len();
        assert_eq!(n, msgs.len());
        assert_eq!(n, key_index.len());
        let sg: Vec<u8> = sigs.iter().flat_map(|s| s.iter().copied()).collect();
        let m = col(n, |i| msg_le32(&msgs[i]));
        let (mut ok, mut st) = (vec![0u8; n], vec![0u8; n]);
        check(unsafe { ffi::bjj_verify_keyset_compressed_batch(engine().raw(), self.ks, n, key_index.as_ptr(), sg.as_ptr(),
                                                               m.as_ptr(), ok.as_mut_ptr(), st.as_mut_ptr()) },
              "bjj_verify_keyset_compressed_batch");
        (0..n).map(|i| if st[i] == 0 { Ok(ok[i] == 1) } else { Err(status_str(st[i])) }).collect()
    }
    /// `verify_schnorr_batch` with pk = keys[key_index[i]], on the compact tables
    pub fn verify_schnorr_batch(&self, key_index: &[u32], msgs: &[BigInt], sigs: &[(Point, BigInt)]) -> Vec<Result<bool, String>> {
        let l = schnorr_lanes(msgs, sigs);
        assert_eq!(l.n, key_index.len());
        let (mut ok, mut st) = (vec![0u8; l.n], vec![0u8; l.n]);
        check(unsafe { ffi::bjj_verify_schnorr_keyset_batch(engine().raw(), self.ks, l.n, key_index.as_ptr(), l.m.as_ptr(),
                                                            l.rx.as_ptr(), l.ry.as_ptr(), l.s.as_ptr(), l.words as i32,
                                                            ok.as_mut_ptr(), st.as_mut_ptr()) }, "bjj_verify_schnorr_keyset_batch");
        schnorr_results(&ok, &st)
    }
    /// the index of each 32-byte compressed key in the set (the smallest if the set holds the point twice), or `None`
    pub fn lookup(&self, pks: &[[u8; 32]]) -> Vec<Option<u32>> {
        let n = pks.len();
        let pk: Vec<u8> = pks.iter().flat_map(|p| p.iter().copied()).collect();
        let mut ki = vec![0u32; n];
        check(unsafe { ffi::bjj_keyset_lookup_batch(engine().raw(), self.ks, n, pk.as_ptr(), ki.as_mut_ptr()) }, "bjj_keyset_lookup_batch");
        ki.into_iter().map(|k| if k == ffi::BJJ_KEY_NONE { None } else { Some(k) }).collect()
    }
    /// `verify_compressed_batch` for keys of the set found by their compressed bytes: `Err` carries R8's decompression
    /// error, `Ok(None)` a key that is not in the set
    pub fn verify_compressed_by_key(&self, pks: &[[u8; 32]], sigs: &[[u8; 64]], msgs: &[BigInt]) -> Vec<Result<Option<bool>, String>> {
        let n = sigs.len();
        assert_eq!(n, msgs.len());
        assert_eq!(n, pks.len());
        let sg: Vec<u8> = sigs.iter().flat_map(|s| s.iter().copied()).collect();
        let pk: Vec<u8> = pks.iter().flat_map(|p| p.iter().copied()).collect();
        let m = col(n, |i| msg_le32(&msgs[i]));
        let (mut ok, mut st, mut ki) = (vec![0u8; n], vec![0u8; n], vec![0u32; n]);
        check(unsafe { ffi::bjj_verify_keyset_lookup_compressed_batch(engine().raw(), self.ks, n, sg.as_ptr(), pk.as_ptr(), m.as_ptr(),
                                                                      ok.as_mut_ptr(), st.as_mut_ptr(), ki.as_mut_ptr()) },
              "bjj_verify_keyset_lookup_compressed_batch");
        (0..n).map(|i| if st[i] != 0 { Err(status_str(st[i])) } else if ki[i] == ffi::BJJ_KEY_NONE { Ok(None) } else { Ok(Some(ok[i] == 1)) })
              .collect()
    }
    /// `[keys[key_index[i]].mul_scalar(k[i])]`
    pub fn mul_batch(&self, key_index: &[u32], scalars: &[BigInt]) -> Vec<Point> {
        let n = scalars.len();
        assert_eq!(n, key_index.len());
        let k = col(n, |i| scalar_base_le32(&scalars[i]));
        let (mut rx, mut ry) = (vec![0u8; 32 * n], vec![0u8; 32 * n]);
        check(unsafe { ffi::bjj_keyset_mul_batch(engine().raw(), self.ks, n, key_index.as_ptr(), k.as_ptr(), rx.as_mut_ptr(),
                                                 ry.as_mut_ptr()) }, "bjj_keyset_mul_batch");
        (0..n).map(|i| Point { x: row(&rx, i), y: row(&ry, i) }).collect()
    }
}
impl Drop for KeySet {
    fn drop(&mut self) {
        unsafe { ffi::bjj_keyset_destroy(engine().raw(), self.ks) }
    }
}

pub fn public_batch(keys: &[PrivateKey]) -> Vec<Point> {
    let n = keys.len();
    let k = col(n, |i| keys[i].key);
    let (mut rx, mut ry) = (vec![0u8; 32 * n], vec![0u8; 32 * n]);
    check(unsafe { ffi::bjj_public_batch(engine().raw(), n, k.as_ptr(), rx.as_mut_ptr(), ry.as_mut_ptr()) },
          "bjj_public_batch");
    (0..n).map(|i| Point { x: row(&rx, i), y: row(&ry, i) }).collect()
}

/// `keys[i].public().compress()` (src/lib.rs:304-306, 166-178) without the affine coordinates crossing PCIe
pub fn public_compressed_batch(keys: &[PrivateKey]) -> Vec<[u8; 32]> {
    let n = keys.len();
    let k = col(n, |i| keys[i].key);
    let mut out = vec![0u8; 32 * n];
    check(unsafe { ffi::bjj_public_compressed_batch(engine().raw(), n, k.as_ptr(), out.as_mut_ptr()) },
          "bjj_public_compressed_batch");
    (0..n).map(|i| row(&out, i)).collect()
}

/// `keys[i].sign(msgs[i]).map(|s| s.compress())` (src/lib.rs:308-342, 245-257); msg > Q gives the reference's Err.
/// Panics on a negative msg, which the reference cannot convert to Fr.
pub fn sign_compressed_batch(keys: &[PrivateKey], msgs: &[BigInt]) -> Vec<Result<[u8; 64], String>> {
    let n = keys.len();
    assert_eq!(n, msgs.len());
    assert!(msgs.iter().all(|m| m.sign() != Sign::Minus), "negative msg");
    let k = col(n, |i| keys[i].key);
    let m = col(n, |i| msg_le32(&msgs[i]));
    let (mut sig, mut st) = (vec![0u8; 64 * n], vec![0u8; n]);
    check(unsafe { ffi::bjj_sign_compressed_batch(engine().raw(), n, k.as_ptr(), m.as_ptr(), sig.as_mut_ptr(),
                                                  st.as_mut_ptr()) }, "bjj_sign_compressed_batch");
    (0..n)
        .map(|i| {
            if st[i] != 0 {
                return Err(status_str(st[i]));
            }
            let mut r = [0u8; 64];
            r.copy_from_slice(&sig[64 * i..64 * i + 64]);
            Ok(r)
        })
        .collect()
}

/// `keys[i].sign_schnorr(msgs[i])` (src/lib.rs:344-362) with the nonce `nonces[i]` instead of the reference's random
/// 1024-bit one: `(r, s)` with `s = k + scalar_key * h` unreduced; msg > Q gives the reference's Err.  The nonces cross
/// the ABI in the smallest multiple of 256 bits that holds the widest.  Panics on a negative msg or nonce, or on a nonce
/// wider than 2048 bits.
pub fn sign_schnorr_batch_with_nonces(keys: &[PrivateKey], msgs: &[BigInt], nonces: &[BigInt]) -> Vec<Result<(Point, BigInt), String>> {
    let n = keys.len();
    assert!(n == msgs.len() && n == nonces.len());
    assert!(msgs.iter().all(|m| m.sign() != Sign::Minus), "negative msg");
    assert!(nonces.iter().all(|k| k.sign() != Sign::Minus), "negative nonce");
    let bits = nonces.iter().map(|k| k.bits()).max().unwrap_or(0).max(1);
    assert!(bits <= 2048, "nonce wider than 2048 bits");
    let words = (8 * ((bits + 255) / 256)) as usize;
    let mut kb = vec![0u8; 4 * words * n];
    for (i, k) in nonces.iter().enumerate() {
        let (_, bytes) = k.to_bytes_le();
        kb[4 * words * i..4 * words * i + bytes.len()].copy_from_slice(&bytes);
    }
    let k = col(n, |i| keys[i].key);
    let m = col(n, |i| msg_le32(&msgs[i]));
    let sw = 4 * (words + 8);
    let (mut rx, mut ry, mut s, mut st) = (vec![0u8; 32 * n], vec![0u8; 32 * n], vec![0u8; sw * n], vec![0u8; n]);
    check(unsafe { ffi::bjj_sign_schnorr_batch(engine().raw(), n, k.as_ptr(), m.as_ptr(), kb.as_ptr(), words as i32, rx.as_mut_ptr(),
                                               ry.as_mut_ptr(), s.as_mut_ptr(), st.as_mut_ptr()) }, "bjj_sign_schnorr_batch");
    (0..n)
        .map(|i| {
            if st[i] != 0 {
                return Err(status_str(st[i]));
            }
            Ok((Point { x: row(&rx, i), y: row(&ry, i) }, BigInt::from_bytes_le(Sign::Plus, &s[sw * i..sw * (i + 1)])))
        })
        .collect()
}

pub fn decompress_batch(blobs: &[[u8; 32]]) -> Vec<Result<Point, String>> {
    let n = blobs.len();
    let inp = col(n, |i| blobs[i]);
    let (mut rx, mut ry, mut st) = (vec![0u8; 32 * n], vec![0u8; 32 * n], vec![0u8; n]);
    check(unsafe { ffi::bjj_decompress_batch(engine().raw(), n, inp.as_ptr(), rx.as_mut_ptr(), ry.as_mut_ptr(),
                                             st.as_mut_ptr()) }, "bjj_decompress_batch");
    (0..n).map(|i| if st[i] == 0 { Ok(Point { x: row(&rx, i), y: row(&ry, i) }) } else { Err(status_str(st[i])) }).collect()
}

pub fn verify_batch(pks: &[Point], sigs: &[Signature], msgs: &[BigInt]) -> Vec<bool> {
    let n = pks.len();
    assert!(n == sigs.len() && n == msgs.len());
    let (r8x, r8y) = (col(n, |i| sigs[i].r_b8.x), col(n, |i| sigs[i].r_b8.y));
    let s = col(n, |i| scalar_b8_le32(&sigs[i].s));
    let (ax, ay) = (col(n, |i| pks[i].x), col(n, |i| pks[i].y));
    let m = col(n, |i| msg_le32(&msgs[i]));
    let mut ok = vec![0u8; n];
    check(unsafe { ffi::bjj_verify_batch(engine().raw(), n, r8x.as_ptr(), r8y.as_ptr(), s.as_ptr(), ax.as_ptr(), ay.as_ptr(),
                                         m.as_ptr(), ok.as_mut_ptr()) }, "bjj_verify_batch");
    ok.into_iter().map(|b| b == 1).collect()
}

// ---- one batch over every device of the box ------------------------------------------------------------

/// `bjj_multi`: one context and one host thread per device inside the library; a call cuts the batch into contiguous
/// shards (BASELINE config 4: 2^24 signatures over 8 GPUs from one caller).  No NCCL: lanes exchange nothing.
pub struct MultiEngine {
    m: *mut ffi::bjj_multi,
}
unsafe impl Send for MultiEngine {}

impl MultiEngine {
    /// all visible devices
    pub fn new() -> Result<MultiEngine, String> {
        let mut m = std::ptr::null_mut();
        let rc = unsafe { ffi::bjj_multi_init(0, std::ptr::null(), &mut m) };
        if rc != ffi::BJJ_OK {
            return Err(format!("bjj_multi_init failed: {}", err_str(rc)));
        }
        Ok(MultiEngine { m })
    }
    pub fn devices(&self) -> i32 {
        unsafe { ffi::bjj_multi_devices(self.m) }
    }
    /// page-lock the caller's (pageable) arrays for the duration of each call
    pub fn set_host_register(&mut self, on: bool) {
        unsafe { ffi::bjj_multi_set_host_register(self.m, on as i32) }
    }
    pub fn verify_batch(&mut self, pks: &[Point], sigs: &[Signature], msgs: &[BigInt]) -> Vec<bool> {
        let n = pks.len();
        assert!(n == sigs.len() && n == msgs.len());
        let (r8x, r8y) = (col(n, |i| sigs[i].r_b8.x), col(n, |i| sigs[i].r_b8.y));
        let s = col(n, |i| scalar_b8_le32(&sigs[i].s));
        let (ax, ay) = (col(n, |i| pks[i].x), col(n, |i| pks[i].y));
        let m = col(n, |i| msg_le32(&msgs[i]));
        let mut ok = vec![0u8; n];
        check(unsafe { ffi::bjj_multi_verify_batch(self.m, n, r8x.as_ptr(), r8y.as_ptr(), s.as_ptr(), ax.as_ptr(), ay.as_ptr(),
                                                   m.as_ptr(), ok.as_mut_ptr()) }, "bjj_multi_verify_batch");
        ok.into_iter().map(|b| b == 1).collect()
    }
    pub fn public_batch(&mut self, keys: &[PrivateKey]) -> Vec<Point> {
        let n = keys.len();
        let k = col(n, |i| keys[i].key);
        let (mut rx, mut ry) = (vec![0u8; 32 * n], vec![0u8; 32 * n]);
        check(unsafe { ffi::bjj_multi_public_batch(self.m, n, k.as_ptr(), rx.as_mut_ptr(), ry.as_mut_ptr()) }, "bjj_multi_public_batch");
        (0..n).map(|i| Point { x: row(&rx, i), y: row(&ry, i) }).collect()
    }
    pub fn public_compressed_batch(&mut self, keys: &[PrivateKey]) -> Vec<[u8; 32]> {
        let n = keys.len();
        let k = col(n, |i| keys[i].key);
        let mut out = vec![0u8; 32 * n];
        check(unsafe { ffi::bjj_multi_public_compressed_batch(self.m, n, k.as_ptr(), out.as_mut_ptr()) },
              "bjj_multi_public_compressed_batch");
        (0..n).map(|i| row(&out, i)).collect()
    }
}
impl Drop for MultiEngine {
    fn drop(&mut self) {
        unsafe { ffi::bjj_multi_destroy(self.m) }
    }
}
