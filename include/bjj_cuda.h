/* libbjj_cuda -- C ABI of the B200-native batch engine for babyjubjub-rs's hot path.
 *
 * The reference crate (arnaucube/babyjubjub-rs) has no FFI of its own; its boundary is the public
 * Rust API.  Each entry point below names the reference item it batches (paths are into the
 * reference tree).  The Rust host crate binds these with `extern "C"` (see INTEGRATION.md); the
 * Python ctypes mirror in babyjubjub-rs_b200/ binds exactly the same symbols.
 *
 * LAYOUT.  Structure-of-arrays.  Every field element, scalar, message and compressed point is 32
 * bytes little-endian; element i of an array lives at byte offset 32*i.  Field elements (point
 * coordinates) are canonical integers < Q, i.e. the bytes of ff_ce's FrRepr([u64;4]) after
 * into_repr().  Scalars and messages are plain 256-bit unsigned integers.  A 64-byte compressed
 * signature is compress(R8) || S_le32 (reference src/lib.rs:245-257), element i at offset 64*i.
 *
 * OWNERSHIP.  The caller owns every buffer passed in.  The library owns device memory, streams and
 * tables inside bjj_ctx; nothing returned must be freed except the ctx (and bjj_host_alloc memory).
 *
 * TWO FLAVOURS per operation:
 *   bjj_<op>_batch      host pointers; copies in, runs, copies out, returns when results are in place.
 *   bjj_<op>_batch_dev  device pointers (16-byte aligned) on the ctx's device; asynchronous on `stream`
 *                       (a cudaStream_t cast to void*; NULL = the ctx's own stream).  Call bjj_sync()
 *                       before reading results or the error flags.
 *
 * ERRORS.  Every function returns 0 on success or one of the BJJ_ERR_* codes.  Per-lane outcomes
 * that the reference reports as Result/Err or bool are per-lane bytes (status / ok arrays).
 * Non-canonical field elements (>= Q) cannot be constructed through the reference's Rust types; at
 * this ABI they are an argument error: the batch still runs with those values reduced mod Q and the
 * call (or the next bjj_sync for _dev calls) returns BJJ_ERR_NONCANONICAL.
 *
 * THREADING.  One bjj_ctx per device, driven by one host thread at a time.  Contexts are
 * independent; there is no global mutable state and no NCCL (nothing is exchanged between lanes).
 *
 * There is NO CPU fallback: bjj_init fails if no CUDA device is usable.
 */
#ifndef BJJ_CUDA_H
#define BJJ_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct bjj_ctx bjj_ctx;

#define BJJ_OK 0
#define BJJ_ERR_CUDA 1          /* a CUDA runtime call failed; see bjj_last_cuda_error() */
#define BJJ_ERR_ARG 2           /* null pointer, bad size, bad input count */
#define BJJ_ERR_NONCANONICAL 3  /* some field-element input was >= Q (results computed mod Q) */
#define BJJ_ERR_NOMEM 4

/* per-lane status bytes of decompress / verify_compressed; 1:1 with the reference's Err strings */
#define BJJ_STATUS_OK 0
#define BJJ_STATUS_Y_RANGE 1     /* "y outside the Finite Field over R"  src/lib.rs:202 */
#define BJJ_STATUS_NO_INV 2      /* "no mod inv of Zero"                 src/utils.rs:14 */
#define BJJ_STATUS_NOT_SQUARE 3  /* "not a mod p square"                 src/utils.rs:119 */
#define BJJ_STATUS_MSG_RANGE 4   /* "msg outside the Finite Field"       src/lib.rs:310 sign, :366 schnorr */

/* Fr test-hook opcodes (bjj_fr_op_batch) */
#define BJJ_FR_MUL 0
#define BJJ_FR_ADD 1
#define BJJ_FR_SUB 2
#define BJJ_FR_INV 3
#define BJJ_FR_SQR 4
#define BJJ_FR_SQR_LAZY 5   /* a^2 computed on (a mod Q) + Q: the squaring on the upper half of the lazy domain */

#define BJJ_POSEIDON_MAX_INPUTS 6   /* poseidon-rs 0.0.8: t = n_inputs + 1 <= 7 */

/* ---- context ------------------------------------------------------------------------------- */
int bjj_device_count(void);
int bjj_init(int device, bjj_ctx** out);      /* builds the B8 comb table on the device */
void bjj_destroy(bjj_ctx* ctx);
int bjj_sync(bjj_ctx* ctx);                   /* waits for the ctx stream; returns and clears pending error flags */
const char* bjj_error_string(int code);       /* static string; for status codes use bjj_status_string */
const char* bjj_status_string(int status);    /* the reference's exact Err text for a lane status */
const char* bjj_last_cuda_error(bjj_ctx* ctx);
void* bjj_stream(bjj_ctx* ctx);               /* the ctx's cudaStream_t */
int bjj_device(bjj_ctx* ctx);
unsigned long long bjj_kernel_launches(bjj_ctx* ctx);   /* kernels launched by this ctx so far */
/* pinned host memory for the host-pointer flavour (plain malloc'd memory also works, slower) */
void* bjj_host_alloc(size_t bytes);
void bjj_host_free(void* p);
/* device memory helpers so a host language without a CUDA binding can use the _dev flavour */
void* bjj_dev_alloc(bjj_ctx* ctx, size_t bytes);
void bjj_dev_free(bjj_ctx* ctx, void* p);
int bjj_memcpy_h2d(bjj_ctx* ctx, void* dst, const void* src, size_t bytes);   /* async on ctx stream */
int bjj_memcpy_d2h(bjj_ctx* ctx, void* dst, const void* src, size_t bytes);   /* async on ctx stream */

/* ---- Fr (reference: `pub type Fr = poseidon_rs::Fr`, src/lib.rs:7) -- test hook ---------------- */
/* out[i] = a[i] (op) b[i] in the field; INV and SQR ignore b (may be NULL -> a is reused) */
int bjj_fr_op_batch(bjj_ctx* ctx, int op, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out);
int bjj_fr_op_batch_dev(bjj_ctx* ctx, int op, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out, void* stream);

/* ---- verify's half-size scalars (no reference counterpart; csrc/split.cuh) -- test hook ---------
 * For every 256-bit h and s:  u = v*h (mod SUBORDER), v odd and non-zero, w = |v|*s (mod SUBORDER).
 * v32 holds |v| with the sign of v in bit 255.  Lets the parity suite drive the device code with crafted h
 * (verify itself only ever sees Poseidon outputs). */
int bjj_split_scalars_batch(bjj_ctx* ctx, size_t n, const uint8_t* h32, const uint8_t* s32, uint8_t* u32, uint8_t* v32,
                            uint8_t* w32);
int bjj_split_scalars_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* h32, const uint8_t* s32, uint8_t* u32,
                                uint8_t* v32, uint8_t* w32, void* stream);

/* ---- PointProjective::add (src/lib.rs:88-131): literal add-2008-bbjlp, projective in and out ---- */
int bjj_add_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz,
                  const uint8_t* qx, const uint8_t* qy, const uint8_t* qz, uint8_t* rx, uint8_t* ry, uint8_t* rz);
int bjj_add_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz,
                      const uint8_t* qx, const uint8_t* qy, const uint8_t* qz, uint8_t* rx, uint8_t* ry,
                      uint8_t* rz, void* stream);

/* ---- PointProjective::affine (src/lib.rs:70-85): (X/Z, Y/Z); Z == 0 -> (0,0) -------------------- */
int bjj_affine_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz,
                     uint8_t* rx, uint8_t* ry);
int bjj_affine_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz,
                         uint8_t* rx, uint8_t* ry, void* stream);

/* ---- Point::mul_scalar (src/lib.rs:149-164): r = |n| * P, n a 256-bit unsigned scalar, unreduced.
 *      Off-curve P is allowed (public fields) and replays the reference sequence bit-exactly. ------ */
int bjj_mul_scalar_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32,
                         uint8_t* rx, uint8_t* ry);
int bjj_mul_scalar_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py,
                             const uint8_t* scalar32, uint8_t* rx, uint8_t* ry, void* stream);

/* The same for BigInt scalars wider than 256 bits (src/lib.rs:149-164 loops over n.bits() of a BigInt of any size):
 * scalar i is `scalar_words` 32-bit little-endian words at byte offset 4*scalar_words*i, 8 <= scalar_words <= 64, a
 * multiple of 8.  On-curve points: the scalar is reduced mod ORDER on the device (exact: their order divides ORDER).
 * Off-curve points: every bit is replayed like the reference does. */
int bjj_mul_scalar_wide_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar,
                              int scalar_words, uint8_t* rx, uint8_t* ry);
int bjj_mul_scalar_wide_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar,
                                  int scalar_words, uint8_t* rx, uint8_t* ry, void* stream);

/* ---- B8.mul_scalar(k) (src/lib.rs:305, :329, :405): fixed-base comb ----------------------------- */
int bjj_fixed_base_batch(bjj_ctx* ctx, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry);
int bjj_fixed_base_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry, void* stream);

/* ---- fixed-base tables for caller-chosen points: P.mul_scalar(k) and k*P + l*Q on the comb path ------
 * A bjj_base is the comb table of one on-curve point P, the same 50 MB of device memory as the context's B8 table,
 * so k*P costs what B8.mul_scalar(k) costs instead of mul_scalar's variable-base ladder.  It pays off for many
 * scalars against one point (commitments m*G + r*H, ElGamal to one recipient, any repeated P.mul_scalar(k_i)).
 *   - bjj_base_create builds the table on the device, synchronously on the ctx stream (one kernel).  The handle
 *     belongs to ctx: it holds device memory of ctx's device until bjj_base_destroy, which must come before
 *     bjj_destroy(ctx).  A call that passes it with another context returns BJJ_ERR_ARG.
 *   - P must be on the curve: an off-curve point returns BJJ_ERR_ARG and *out = NULL.  (The reference's result for
 *     an off-curve point depends on its exact double-and-add order, which no table reproduces; such callers keep
 *     bjj_mul_scalar_batch, which replays it.)  A coordinate >= Q returns BJJ_ERR_NONCANONICAL and no handle.
 *   - Scalars are raw 256-bit values, unreduced, like bjj_fixed_base_batch's: every on-curve point has an order
 *     dividing ORDER, so every k (0, >= ORDER, points with a torsion component) gives the reference's result.
 *   - base == NULL (p / q == NULL) selects the context's B8 table. */
typedef struct bjj_base bjj_base;
int bjj_base_create(bjj_ctx* ctx, const uint8_t* px32, const uint8_t* py32, bjj_base** out);
void bjj_base_destroy(bjj_ctx* ctx, bjj_base* base);   /* waits for the device, then frees; NULL is a no-op */
/* r = k*P  (Point::mul_scalar, src/lib.rs:149-164) */
int bjj_base_mul_batch(bjj_ctx* ctx, const bjj_base* base, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry);
int bjj_base_mul_batch_dev(bjj_ctx* ctx, const bjj_base* base, size_t n, const uint8_t* scalar32, uint8_t* rx,
                           uint8_t* ry, void* stream);
/* r = (k*P).projective().add((l*Q).projective()).affine()  (src/lib.rs:70-131, 149-164) */
int bjj_base_mul2_batch(bjj_ctx* ctx, const bjj_base* p, const bjj_base* q, size_t n, const uint8_t* k32,
                        const uint8_t* l32, uint8_t* rx, uint8_t* ry);
int bjj_base_mul2_batch_dev(bjj_ctx* ctx, const bjj_base* p, const bjj_base* q, size_t n, const uint8_t* k32,
                            const uint8_t* l32, uint8_t* rx, uint8_t* ry, void* stream);

/* ---- PrivateKey::public (src/lib.rs:304-306) = B8 * scalar_key(key);  scalar_key (:284-302) ------ */
int bjj_public_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* rx, uint8_t* ry);
int bjj_public_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* rx, uint8_t* ry, void* stream);
/* compress(PrivateKey::public(key)) (src/lib.rs:304-306, 166-178): 32 B per lane, the same bytes as bjj_public_batch
 * followed by bjj_compress_batch, without the affine coordinates crossing PCIe.  Runs the kernels of bjj_public_batch
 * (BJJ_PUBLIC_FUSED selects the same path) with a compressing last pass. */
int bjj_public_compressed_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* out32);
int bjj_public_compressed_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* out32, void* stream);
int bjj_scalar_key_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* scalar32);
int bjj_scalar_key_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* scalar32, void* stream);

/* ---- PrivateKey::sign (src/lib.rs:308-342): deterministic EdDSA-Poseidon signing ("next" row: the
 *      caller-side producer of verify's inputs; also the device-side fixture generator of bench.py).
 *      status[i] = 0, or BJJ_STATUS_MSG_RANGE when msg > Q (outputs zero). ------------------------- */
int bjj_sign_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* r8x, uint8_t* r8y,
                   uint8_t* s32, uint8_t* status);
int bjj_sign_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* r8x,
                       uint8_t* r8y, uint8_t* s32, uint8_t* status, void* stream);
/* PrivateKey::sign(msg).compress() (src/lib.rs:308-342, 245-257): sig64[i] = compress(R8) || S;
 * status[i] = BJJ_STATUS_MSG_RANGE when msg > Q, and then sig64[i] is 64 zero bytes.  Always the kernel pipeline:
 * BJJ_SIGN_FUSED selects the fused kernel for bjj_sign_batch only. */
int bjj_sign_compressed_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* sig64,
                              uint8_t* status);
int bjj_sign_compressed_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* sig64,
                                  uint8_t* status, void* stream);

/* ---- Point::compress (src/lib.rs:166-178) / decompress_point (src/lib.rs:192-224) ---------------- */
int bjj_compress_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, uint8_t* out32);
int bjj_compress_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, uint8_t* out32, void* stream);
/* status[i] != 0 -> rx/ry[i] are zero */
int bjj_decompress_batch(bjj_ctx* ctx, size_t n, const uint8_t* in32, uint8_t* rx, uint8_t* ry, uint8_t* status);
int bjj_decompress_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* in32, uint8_t* rx, uint8_t* ry,
                             uint8_t* status, void* stream);

/* ---- POSEIDON.hash (poseidon-rs 0.0.8 behind src/lib.rs:59,333,370,401): n_inputs in 1..BJJ_POSEIDON_MAX_INPUTS --
 *      the widths that crate accepts (its hash() returns Err("Wrong inputs length") for 0 or more than 6 inputs);
 *      other counts return BJJ_ERR_ARG,
 *      in[j] = array of the j-th input of every lane (host flavour: host array of host pointers;
 *      dev flavour: host array of device pointers). ------------------------------------------------ */
int bjj_poseidon_batch(bjj_ctx* ctx, int n_inputs, size_t n, const uint8_t* const* in, uint8_t* out);
int bjj_poseidon_batch_dev(bjj_ctx* ctx, int n_inputs, size_t n, const uint8_t* const* in, uint8_t* out, void* stream);

/* ---- verify (src/lib.rs:395-412): ok[i] = 1 iff S*B8 == R8 + (8*hm)*A, hm = Poseidon(R8,A,msg);
 *      msg > Q -> 0.  No range check on S, no subgroup check on A / R8 (reference semantics). -------- */
int bjj_verify_batch(bjj_ctx* ctx, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32,
                     const uint8_t* ax, const uint8_t* ay, const uint8_t* msg32, uint8_t* ok);
int bjj_verify_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32,
                         const uint8_t* ax, const uint8_t* ay, const uint8_t* msg32, uint8_t* ok, void* stream);

/* ---- verify_schnorr (src/lib.rs:375-385) with schnorr_hash (src/lib.rs:364-373):
 *      ok[i] = 1 iff s*B8 == r + h*pk, h = Poseidon(pk.x, pk.y, r.x, r.y, msg); status[i] = BJJ_STATUS_MSG_RANGE
 *      (the reference's Err("msg outside the Finite Field")) when msg > Q.  s is 256-bit: the reference's s =
 *      k + x*h is an unreduced ~1024-bit BigInt, which the host reduces mod SUBORDER (B8 has that order). ---- */
int bjj_verify_schnorr_batch(bjj_ctx* ctx, size_t n, const uint8_t* pkx, const uint8_t* pky, const uint8_t* msg32,
                             const uint8_t* rx, const uint8_t* ry, const uint8_t* s32, uint8_t* ok, uint8_t* status);
int bjj_verify_schnorr_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* pkx, const uint8_t* pky, const uint8_t* msg32,
                                 const uint8_t* rx, const uint8_t* ry, const uint8_t* s32, uint8_t* ok, uint8_t* status,
                                 void* stream);

/* ---- decompress_signature + decompress_point(pk) + verify (src/lib.rs:260-268, 192-224, 395-412):
 *      status[i] = first decompression error (R8 first, then A); ok[i] = 0 whenever status[i] != 0. -- */
int bjj_verify_compressed_batch(bjj_ctx* ctx, size_t n, const uint8_t* sig64, const uint8_t* pk32,
                                const uint8_t* msg32, uint8_t* ok, uint8_t* status);
int bjj_verify_compressed_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* sig64, const uint8_t* pk32,
                                    const uint8_t* msg32, uint8_t* ok, uint8_t* status, void* stream);

/* ---- multi-device: ONE caller, ONE host batch, N devices of one box -------------------------------
 * BASELINE.json config 4 as written (2^24 signatures across 8 B200 from one caller).  The reference has no
 * counterpart (it is single-threaded: src/lib.rs:395-412 verifies one signature); a rayon par_iter over a
 * batch is what this replaces.  A bjj_multi owns one bjj_ctx and one persistent host thread per device; a call
 * cuts the arrays into contiguous shards (lane i of shard d is lane n*d/N + i of the batch), runs the ordinary
 * host-pointer entry point on every shard concurrently and returns when all are done.  No NCCL, no peer access:
 * nothing is exchanged between lanes.  Arrays may be pageable or pinned (bjj_host_alloc); with
 * bjj_multi_set_host_register(m, 1) pageable arrays are page-locked for the duration of each call. */
typedef struct bjj_multi bjj_multi;
int bjj_multi_init(int n_devices, const int* devices, bjj_multi** out);   /* n_devices <= 0: all; devices NULL: 0..n-1 */
void bjj_multi_destroy(bjj_multi* m);
int bjj_multi_devices(bjj_multi* m);
bjj_ctx* bjj_multi_ctx(bjj_multi* m, int i);                              /* the context of device slot i */
void bjj_multi_set_host_register(bjj_multi* m, int on);
unsigned long long bjj_multi_kernel_launches(bjj_multi* m);
int bjj_multi_verify_batch(bjj_multi* m, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32,
                           const uint8_t* ax, const uint8_t* ay, const uint8_t* msg32, uint8_t* ok);
int bjj_multi_verify_compressed_batch(bjj_multi* m, size_t n, const uint8_t* sig64, const uint8_t* pk32,
                                      const uint8_t* msg32, uint8_t* ok, uint8_t* status);
int bjj_multi_mul_scalar_batch(bjj_multi* m, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32,
                               uint8_t* rx, uint8_t* ry);
int bjj_multi_public_batch(bjj_multi* m, size_t n, const uint8_t* key32, uint8_t* rx, uint8_t* ry);
int bjj_multi_public_compressed_batch(bjj_multi* m, size_t n, const uint8_t* key32, uint8_t* out32);
int bjj_multi_sign_compressed_batch(bjj_multi* m, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* sig64,
                                    uint8_t* status);
int bjj_multi_fixed_base_batch(bjj_multi* m, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry);
int bjj_multi_decompress_batch(bjj_multi* m, size_t n, const uint8_t* in32, uint8_t* rx, uint8_t* ry, uint8_t* status);

#ifdef __cplusplus
}
#endif
#endif /* BJJ_CUDA_H */
