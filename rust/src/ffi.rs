//! `extern "C"` declarations for include/bjj_cuda.h, one per exported symbol.
//! Each comment names the reference item (arnaucube/babyjubjub-rs) the entry point batches.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

#[repr(C)]
pub struct bjj_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct bjj_base {
    _private: [u8; 0],
}
#[repr(C)]
pub struct bjj_multi {
    _private: [u8; 0],
}

pub const BJJ_OK: c_int = 0;
pub const BJJ_ERR_CUDA: c_int = 1;
pub const BJJ_ERR_ARG: c_int = 2;
pub const BJJ_ERR_NONCANONICAL: c_int = 3;
pub const BJJ_ERR_NOMEM: c_int = 4;

extern "C" {
    pub fn bjj_device_count() -> c_int;
    pub fn bjj_init(device: c_int, out: *mut *mut bjj_ctx) -> c_int;
    pub fn bjj_destroy(ctx: *mut bjj_ctx);
    pub fn bjj_sync(ctx: *mut bjj_ctx) -> c_int;
    pub fn bjj_error_string(code: c_int) -> *const c_char;
    pub fn bjj_status_string(status: c_int) -> *const c_char;
    pub fn bjj_last_cuda_error(ctx: *mut bjj_ctx) -> *const c_char;
    pub fn bjj_stream(ctx: *mut bjj_ctx) -> *mut c_void;
    pub fn bjj_device(ctx: *mut bjj_ctx) -> c_int;
    pub fn bjj_kernel_launches(ctx: *mut bjj_ctx) -> u64;
    pub fn bjj_host_alloc(bytes: usize) -> *mut c_void;
    pub fn bjj_host_free(p: *mut c_void);
    pub fn bjj_dev_alloc(ctx: *mut bjj_ctx, bytes: usize) -> *mut c_void;
    pub fn bjj_dev_free(ctx: *mut bjj_ctx, p: *mut c_void);
    pub fn bjj_memcpy_h2d(ctx: *mut bjj_ctx, dst: *mut c_void, src: *const c_void, bytes: usize) -> c_int;
    pub fn bjj_memcpy_d2h(ctx: *mut bjj_ctx, dst: *mut c_void, src: *const c_void, bytes: usize) -> c_int;

    // Fr ops (src/lib.rs:7) -- test hook
    pub fn bjj_fr_op_batch(ctx: *mut bjj_ctx, op: c_int, n: usize, a: *const u8, b: *const u8, out: *mut u8) -> c_int;
    pub fn bjj_split_scalars_batch(ctx: *mut bjj_ctx, n: usize, h32: *const u8, s32: *const u8, u32_: *mut u8, v32: *mut u8,
                                   w32: *mut u8) -> c_int;
    // PointProjective::add (src/lib.rs:88-131)
    pub fn bjj_add_batch(ctx: *mut bjj_ctx, n: usize, px: *const u8, py: *const u8, pz: *const u8, qx: *const u8,
                         qy: *const u8, qz: *const u8, rx: *mut u8, ry: *mut u8, rz: *mut u8) -> c_int;
    // PointProjective::affine (src/lib.rs:70-85)
    pub fn bjj_affine_batch(ctx: *mut bjj_ctx, n: usize, px: *const u8, py: *const u8, pz: *const u8, rx: *mut u8,
                            ry: *mut u8) -> c_int;
    // Point::mul_scalar (src/lib.rs:149-164)
    pub fn bjj_mul_scalar_batch(ctx: *mut bjj_ctx, n: usize, px: *const u8, py: *const u8, scalar32: *const u8,
                                rx: *mut u8, ry: *mut u8) -> c_int;
    // the same for BigInt scalars wider than 256 bits (scalar_words x 32-bit words per lane)
    pub fn bjj_mul_scalar_wide_batch(ctx: *mut bjj_ctx, n: usize, px: *const u8, py: *const u8, scalar: *const u8,
                                     scalar_words: c_int, rx: *mut u8, ry: *mut u8) -> c_int;
    // B8.mul_scalar (src/lib.rs:305,329,405)
    pub fn bjj_fixed_base_batch(ctx: *mut bjj_ctx, n: usize, scalar32: *const u8, rx: *mut u8, ry: *mut u8) -> c_int;
    // comb table of a caller-chosen on-curve point (50 MB of device memory, owned by ctx); NULL base = B8
    pub fn bjj_base_create(ctx: *mut bjj_ctx, px32: *const u8, py32: *const u8, out: *mut *mut bjj_base) -> c_int;
    pub fn bjj_base_destroy(ctx: *mut bjj_ctx, base: *mut bjj_base);
    // P.mul_scalar(k) (src/lib.rs:149-164) on the table of P
    pub fn bjj_base_mul_batch(ctx: *mut bjj_ctx, base: *const bjj_base, n: usize, scalar32: *const u8, rx: *mut u8,
                              ry: *mut u8) -> c_int;
    // (k*P).projective().add((l*Q).projective()).affine() (src/lib.rs:70-131, 149-164)
    pub fn bjj_base_mul2_batch(ctx: *mut bjj_ctx, p: *const bjj_base, q: *const bjj_base, n: usize, k32: *const u8,
                               l32: *const u8, rx: *mut u8, ry: *mut u8) -> c_int;
    // PrivateKey::public / scalar_key / sign (src/lib.rs:284-342)
    pub fn bjj_public_batch(ctx: *mut bjj_ctx, n: usize, key32: *const u8, rx: *mut u8, ry: *mut u8) -> c_int;
    pub fn bjj_scalar_key_batch(ctx: *mut bjj_ctx, n: usize, key32: *const u8, scalar32: *mut u8) -> c_int;
    pub fn bjj_sign_batch(ctx: *mut bjj_ctx, n: usize, key32: *const u8, msg32: *const u8, r8x: *mut u8, r8y: *mut u8,
                          s32: *mut u8, status: *mut u8) -> c_int;
    // compress(PrivateKey::public) / PrivateKey::sign(msg).compress() (src/lib.rs:166-178, 245-257, 304-342)
    pub fn bjj_public_compressed_batch(ctx: *mut bjj_ctx, n: usize, key32: *const u8, out32: *mut u8) -> c_int;
    pub fn bjj_sign_compressed_batch(ctx: *mut bjj_ctx, n: usize, key32: *const u8, msg32: *const u8, sig64: *mut u8,
                                     status: *mut u8) -> c_int;
    // Point::compress / decompress_point (src/lib.rs:166-178, 192-224)
    pub fn bjj_compress_batch(ctx: *mut bjj_ctx, n: usize, px: *const u8, py: *const u8, out32: *mut u8) -> c_int;
    pub fn bjj_decompress_batch(ctx: *mut bjj_ctx, n: usize, in32: *const u8, rx: *mut u8, ry: *mut u8,
                                status: *mut u8) -> c_int;
    // POSEIDON.hash (src/lib.rs:400-401)
    pub fn bjj_poseidon_batch(ctx: *mut bjj_ctx, n_inputs: c_int, n: usize, inputs: *const *const u8, out: *mut u8) -> c_int;
    // verify (src/lib.rs:395-412)
    pub fn bjj_verify_batch(ctx: *mut bjj_ctx, n: usize, r8x: *const u8, r8y: *const u8, s32: *const u8, ax: *const u8,
                            ay: *const u8, msg32: *const u8, ok: *mut u8) -> c_int;
    // verify_schnorr + schnorr_hash (src/lib.rs:364-385)
    pub fn bjj_verify_schnorr_batch(ctx: *mut bjj_ctx, n: usize, pkx: *const u8, pky: *const u8, msg32: *const u8,
                                    rx: *const u8, ry: *const u8, s32: *const u8, ok: *mut u8, status: *mut u8) -> c_int;
    // decompress_signature + decompress_point + verify (src/lib.rs:260-268)
    pub fn bjj_verify_compressed_batch(ctx: *mut bjj_ctx, n: usize, sig64: *const u8, pk32: *const u8,
                                       msg32: *const u8, ok: *mut u8, status: *mut u8) -> c_int;

    // one caller, one host batch, N devices (BASELINE config 4); no reference counterpart
    pub fn bjj_multi_init(n_devices: c_int, devices: *const c_int, out: *mut *mut bjj_multi) -> c_int;
    pub fn bjj_multi_destroy(m: *mut bjj_multi);
    pub fn bjj_multi_devices(m: *mut bjj_multi) -> c_int;
    pub fn bjj_multi_ctx(m: *mut bjj_multi, i: c_int) -> *mut bjj_ctx;
    pub fn bjj_multi_set_host_register(m: *mut bjj_multi, on: c_int);
    pub fn bjj_multi_kernel_launches(m: *mut bjj_multi) -> u64;
    pub fn bjj_multi_verify_batch(m: *mut bjj_multi, n: usize, r8x: *const u8, r8y: *const u8, s32: *const u8, ax: *const u8,
                                  ay: *const u8, msg32: *const u8, ok: *mut u8) -> c_int;
    pub fn bjj_multi_verify_compressed_batch(m: *mut bjj_multi, n: usize, sig64: *const u8, pk32: *const u8, msg32: *const u8,
                                             ok: *mut u8, status: *mut u8) -> c_int;
    pub fn bjj_multi_mul_scalar_batch(m: *mut bjj_multi, n: usize, px: *const u8, py: *const u8, scalar32: *const u8,
                                      rx: *mut u8, ry: *mut u8) -> c_int;
    pub fn bjj_multi_public_batch(m: *mut bjj_multi, n: usize, key32: *const u8, rx: *mut u8, ry: *mut u8) -> c_int;
    pub fn bjj_multi_public_compressed_batch(m: *mut bjj_multi, n: usize, key32: *const u8, out32: *mut u8) -> c_int;
    pub fn bjj_multi_sign_compressed_batch(m: *mut bjj_multi, n: usize, key32: *const u8, msg32: *const u8, sig64: *mut u8,
                                           status: *mut u8) -> c_int;
    pub fn bjj_multi_fixed_base_batch(m: *mut bjj_multi, n: usize, scalar32: *const u8, rx: *mut u8, ry: *mut u8) -> c_int;
    pub fn bjj_multi_decompress_batch(m: *mut bjj_multi, n: usize, in32: *const u8, rx: *mut u8, ry: *mut u8,
                                      status: *mut u8) -> c_int;
}
