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
/* verify (src/lib.rs:395-412) of n signatures made by ONE key A, the point of pk: ok[i] = 1 iff
 * S*B8 == R8 + (8*hm)*A, hm = Poseidon(R8.x, R8.y, A.x, A.y, msg); msg > Q -> 0 (msg == Q hashes as 0).  The same
 * results as bjj_verify_batch with A in every lane, from two comb walks per lane (S against B8's table, 8*hm mod ORDER
 * against pk's) instead of the per-lane window tables and 4 doublings per window.  S is raw 256-bit, unreduced.
 * R8 off the curve replays the reference's sum literally.  A coordinate of R8 >= Q returns BJJ_ERR_NONCANONICAL
 * (the batch is computed mod Q).  pk == NULL or a handle of another context returns BJJ_ERR_ARG: unlike
 * bjj_base_mul, NULL does not select B8 here. */
int bjj_verify_base_batch(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* r8x, const uint8_t* r8y,
                          const uint8_t* s32, const uint8_t* msg32, uint8_t* ok);
int bjj_verify_base_batch_dev(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* r8x, const uint8_t* r8y,
                              const uint8_t* s32, const uint8_t* msg32, uint8_t* ok, void* stream);
/* the same from 64-byte compressed signatures (decompress_signature, src/lib.rs:260-268): status[i] = R8's
 * decompression error (the codes of bjj_verify_compressed_batch), and ok[i] = 0 whenever status[i] != 0.  There is
 * no status for A: bjj_base_create checked it. */
int bjj_verify_base_compressed_batch(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* sig64,
                                     const uint8_t* msg32, uint8_t* ok, uint8_t* status);
int bjj_verify_base_compressed_batch_dev(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* sig64,
                                         const uint8_t* msg32, uint8_t* ok, uint8_t* status, void* stream);

/* ---- key sets: many known keys, each with a compact comb; a key per lane ------------------------------------
 * A bjj_keyset holds n_keys on-curve public keys, each with a table of 8-bit windows (4,130 entries, 396,480 B per
 * key: 65,536 keys take 26 GB) instead of bjj_base's 50 MB, so a batch may mix many keys.  Calls name the key of lane i
 * by key_index[i] (little-endian uint32).  k*P costs 33 mixed additions and no doubling.
 *   - bjj_keyset_create copies the SoA coordinates ax, ay (32 B per key) and builds the tables on the device,
 *     synchronously on the ctx stream.  No handle comes back when: a coordinate is >= Q (BJJ_ERR_NONCANONICAL, which
 *     outranks the next), a key is off the curve (BJJ_ERR_ARG, for the reason given for bjj_base_create), n_keys is 0
 *     or above 2^32 - 1 or a pointer is NULL (BJJ_ERR_ARG), or the tables do not fit in device memory (BJJ_ERR_NOMEM,
 *     with the CUDA error cleared).  key_status (may be NULL) receives one BJJ_KEY_* code per key.
 *   - The handle belongs to ctx like a bjj_base: bjj_keyset_destroy must come before bjj_destroy(ctx), and a call that
 *     passes it with another context returns BJJ_ERR_ARG.
 *   - key_index[i] >= n_keys: that lane gets ok = 0 (status 0 in the compressed form; the point (0, 0) in
 *     bjj_keyset_mul), the other lanes are computed, and the call returns BJJ_ERR_ARG (a _dev call: the next bjj_sync,
 *     where BJJ_ERR_ARG outranks BJJ_ERR_NONCANONICAL). */
typedef struct bjj_keyset bjj_keyset;
#define BJJ_KEY_OK 0            /* key_status codes; the same values as BJJ_BASE_* */
#define BJJ_KEY_OFF_CURVE 1
#define BJJ_KEY_NONCANONICAL 2
int bjj_keyset_create(bjj_ctx* ctx, size_t n_keys, const uint8_t* ax, const uint8_t* ay, uint8_t* key_status,
                      bjj_keyset** out);
void bjj_keyset_destroy(bjj_ctx* ctx, bjj_keyset* ks);   /* waits for the device, then frees; NULL is a no-op */
/* Editing a set in place.  bjj_keyset_append adds n_new keys (SoA, 32 B per coordinate) under the indices n_keys ..
 * n_keys + n_new - 1; bjj_keyset_replace gives keys first .. first + count - 1 new coordinates (key rotation).
 *   - Each new key is checked as by bjj_keyset_create: key_status (may be NULL) receives one BJJ_KEY_* code per new key,
 *     a coordinate >= Q returns BJJ_ERR_NONCANONICAL, which outranks an off-curve key's BJJ_ERR_ARG.
 *   - All or nothing: on any error the set is unchanged (size, tables, lookups), BJJ_ERR_NOMEM included, which also
 *     clears the CUDA error.  (A CUDA fault while replace rebuilds tables in place is the exception: the device is
 *     then unusable anyway.)
 *   - BJJ_ERR_ARG, with nothing allocated: a NULL handle or one of another context, n_keys + n_new > 2^32 - 1
 *     (BJJ_KEY_NONE stays reserved), first + count > n_keys (or an overflow in that sum), then a NULL ax or ay.  After
 *     the first three checks, n_new == 0 or count == 0 returns BJJ_OK and does nothing.
 *   - Synchronous, like create and destroy: both synchronise the device before they touch the set (_dev calls on
 *     other streams may still read it) and return when it is ready.  The handle does not change.
 *   - Existing indices keep their keys under append; replace changes only the replaced ones.  Afterwards every call
 *     on the set returns byte for byte what it returns on a set created from the current key list: a point held twice
 *     is found at its smallest index, x = 0 keys are not indexed, a replaced key's old bytes are no longer found unless
 *     another key holds them.
 *   - Address space: every set reserves GPU virtual address space for total device memory / 396,480 B tables
 *     (191.5 GB on a 180 GB B200), so a process holds a few hundred sets at most (733 one-key sets were measured);
 *     past that, bjj_keyset_create returns BJJ_ERR_NOMEM.
 *   - Cost: the new or replaced keys only (1 + 2 * ceil(n / 511) kernel launches, as create of n keys), plus a host
 *     rebuild of the lookup index.  The tables grow inside an address range reserved by create, so an append never
 *     copies them: device memory peaks at the final set plus the build's scratch. */
int bjj_keyset_append(bjj_ctx* ctx, bjj_keyset* ks, size_t n_new, const uint8_t* ax, const uint8_t* ay,
                      uint8_t* key_status);
int bjj_keyset_replace(bjj_ctx* ctx, bjj_keyset* ks, size_t first, size_t count, const uint8_t* ax, const uint8_t* ay,
                       uint8_t* key_status);
/* verify (src/lib.rs:395-412) with A = key key_index[i] of ks: byte for byte bjj_verify_batch with those keys in ax, ay
 * (msg > Q -> 0, msg == Q hashes as 0, S raw and unreduced, torsion components accepted, R8 off the curve replayed
 * literally, an R8 coordinate >= Q -> BJJ_ERR_NONCANONICAL), from two comb walks per lane like bjj_verify_base_batch */
int bjj_verify_keyset_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* r8x,
                            const uint8_t* r8y, const uint8_t* s32, const uint8_t* msg32, uint8_t* ok);
int bjj_verify_keyset_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* r8x,
                                const uint8_t* r8y, const uint8_t* s32, const uint8_t* msg32, uint8_t* ok, void* stream);
/* the same from 64-byte signatures (decompress_signature, src/lib.rs:260-268): status[i] = R8's decompression error */
int bjj_verify_keyset_compressed_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index,
                                       const uint8_t* sig64, const uint8_t* msg32, uint8_t* ok, uint8_t* status);
int bjj_verify_keyset_compressed_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index,
                                           const uint8_t* sig64, const uint8_t* msg32, uint8_t* ok, uint8_t* status,
                                           void* stream);
/* r_i = P_{key_index[i]}.mul_scalar(k_i) (src/lib.rs:149-164), k raw 256-bit and unreduced, as bjj_base_mul_batch */
int bjj_keyset_mul_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* scalar32,
                         uint8_t* rx, uint8_t* ry);
int bjj_keyset_mul_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* scalar32,
                             uint8_t* rx, uint8_t* ry, void* stream);
/* Keys by their compressed bytes.  bjj_keyset_create also indexes the set by compress(P_j) (src/lib.rs:166-178), on the
 * host: 32 B plus at most 16 B of device memory per key, freed by bjj_keyset_destroy.  The index's hash is keyed with a
 * seed drawn per set, so chosen keys cannot crowd one probe chain; results do not depend on it.
 *   - bjj_keyset_lookup_batch: key_index[i] = the index j of the key with compress(P_j) == pk32[i], the smallest such j
 *     if the set holds a point twice, else BJJ_KEY_NONE.  A miss is data, not an error.  P and -P (same y, bit 255
 *     apart) are each found under their own index.  The keys with x = 0, (0, 1) and (0, Q-1), are not indexed and come
 *     back BJJ_KEY_NONE: decompress_point rejects their compressed forms (src/utils.rs:118), so no lane of
 *     bjj_verify_compressed_batch verifies against them.  One kernel launch per sub-batch of 2^21 lanes.
 *   - bjj_verify_keyset_lookup_compressed_batch: decompress_signature + decompress_point(pk) + verify (src/lib.rs:260-268,
 *     192-224, 395-412) for keys of ks found by their compressed bytes; the same arrays as bjj_verify_compressed_batch,
 *     and key_index receives the lookup above.  A found lane's ok[i] and status[i] are byte for byte those of
 *     bjj_verify_compressed_batch on the same (sig64, pk32, msg32).  Any other lane gets ok[i] = 0, status[i] = R8's
 *     decompression status and key_index[i] = BJJ_KEY_NONE, with no error code from the call or from the next
 *     bjj_sync.  Six kernel launches per sub-batch: R8's decompression (3), the lookup, then the two kernels of
 *     bjj_verify_keyset_compressed_batch.
 * A NULL pointer, a NULL handle or a handle of another context returns BJJ_ERR_ARG; n == 0 is a no-op. */
#define BJJ_KEY_NONE 0xFFFFFFFFu   /* key_index output of the lookup calls: no key of the set has these bytes */
int bjj_keyset_lookup_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* pk32, uint32_t* key_index);
int bjj_keyset_lookup_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* pk32, uint32_t* key_index,
                                void* stream);
int bjj_verify_keyset_lookup_compressed_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* sig64,
                                              const uint8_t* pk32, const uint8_t* msg32, uint8_t* ok, uint8_t* status,
                                              uint32_t* key_index);
int bjj_verify_keyset_lookup_compressed_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* sig64,
                                                  const uint8_t* pk32, const uint8_t* msg32, uint8_t* ok, uint8_t* status,
                                                  uint32_t* key_index, void* stream);

/* ---- multi-scalar product: R = sum_i P_i.mul_scalar(k_i), one point for the whole batch ----------------------------
 * The reference has no such call; its composition is the fold, in index order,
 *     acc = (0 : 1 : 1);  for i: acc = acc.add(P_i.mul_scalar(k_i).projective());  R = acc.affine()
 * (src/lib.rs:70-131, :149-164).  For points on the curve every P_i.mul_scalar(k_i) is the group element k_i * P_i (the
 * order of an on-curve point divides ORDER, so the raw 256-bit k_i serves as is: 0, values >= ORDER and points with a
 * torsion component included) and PointProjective::add is the complete group law (a is a square, d is not), so R does
 * not depend on how the sum is computed and these calls return the fold's bytes.  Uses: Pedersen vector commitments
 * sum m_i * G_i, weighted sums of ElGamal ciphertexts, batch checks built from random linear combinations.
 *   - Inputs: SoA arrays of n 32-byte little-endian values; scalars raw 256-bit and unreduced (as bjj_base_mul_batch).
 *     Output: ONE canonical affine point, 32 bytes in rx32 and 32 in ry32 (device pointers in _dev).  n == 0 and every
 *     cancelling sum give the identity (0, 1).
 *   - point_status (may be NULL) gets one BJJ_KEY_* code per point.  A point off the curve (the reference's fold past
 *     it is no group law, and no bucket method reproduces its operation sequence) makes the result (0, 0), which is no
 *     curve point, and the call returns BJJ_ERR_ARG; _dev returns it from the next bjj_sync (BJJ_ERR_ARG outranks
 *     BJJ_ERR_NONCANONICAL there).  A coordinate >= Q: the sum is computed mod Q and the call returns
 *     BJJ_ERR_NONCANONICAL.  A NULL ctx, input or output pointer returns BJJ_ERR_ARG; a failed scratch allocation
 *     BJJ_ERR_NOMEM with the CUDA error cleared.
 *   - Device memory: a bucket array of (256/c + 1) x 2^(c-1) points of 128 B (c = 8 below 2^20 points, else 16: 71 MB)
 *     and about 0.5 KB (c = 16) or 0.9 KB (c = 8) per point of a sub-batch of up to 2^20 points, grown on demand and
 *     kept by the context.
 *   - The launch count depends on n only.  The host flavour streams its chunks into the same buckets and synchronises;
 *     _dev is asynchronous on `stream`. */
int bjj_msm_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32, uint8_t* rx32,
                  uint8_t* ry32, uint8_t* point_status);
int bjj_msm_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32, uint8_t* rx32,
                      uint8_t* ry32, uint8_t* point_status, void* stream);

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

/* ---- PrivateKey::sign_schnorr (src/lib.rs:344-362) with the nonce k supplied by the caller (the reference draws
 *      gen_biguint(1024)): r = B8*k, h = schnorr_hash(pk, msg, r) = Poseidon(pk.x, pk.y, r.x, r.y, msg) (src/lib.rs:364-373),
 *      s = k + scalar_key(key)*h, NOT reduced, exactly the reference's BigInt.
 *      Nonce i is `nonce_words` little-endian 32-bit words at byte offset 4*nonce_words*i, nonce_words a multiple of 8 in
 *      8..64 (as bjj_mul_scalar_wide_batch; the reference's 1024-bit nonce is nonce_words = 32); other widths return
 *      BJJ_ERR_ARG.  s[i] is nonce_words + 8 words at byte offset 4*(nonce_words + 8)*i, which always holds it
 *      (scalar_key < 2^252, h < Q < 2^254).  r is (0, 1) for k = 0 and every multiple of SUBORDER, as in the reference.
 *      status[i] = BJJ_STATUS_MSG_RANGE when msg > Q (Err("msg outside the Finite Field")), and then rx, ry and s of the
 *      lane are zero; msg == Q hashes as 0. */
int bjj_sign_schnorr_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, const uint8_t* nonce,
                           int nonce_words, uint8_t* rx, uint8_t* ry, uint8_t* s, uint8_t* status);
int bjj_sign_schnorr_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, const uint8_t* nonce,
                               int nonce_words, uint8_t* rx, uint8_t* ry, uint8_t* s, uint8_t* status, void* stream);

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

/* ---- verify_schnorr (src/lib.rs:364-385) on the signer's own output: s at the width bjj_sign_schnorr_batch writes it.
 *      s[i] is s_words little-endian 32-bit words at byte offset 4*s_words*i: exactly bjj_sign_schnorr_batch's s with
 *      s_words = nonce_words + 8.  s_words a multiple of 8 in 8..72, else BJJ_ERR_ARG.  s is reduced mod SUBORDER on the
 *      device (B8 has that order, so B8.mul_scalar(s) is unchanged).  status[i] = BJJ_STATUS_MSG_RANGE iff msg > Q (then
 *      ok[i] = 0), for every lane; msg == Q hashes as 0.  An r coordinate >= Q returns BJJ_ERR_NONCANONICAL (the batch
 *      is computed mod Q).
 *   - _base: every lane's pk is the key of `pk` (bjj_base_create), on the comb path of bjj_verify_base_batch: one
 *     Poseidon and two comb walks per lane.  pk == NULL or a handle of another context returns BJJ_ERR_ARG.
 *   - _keyset: pk = key key_index[i] of ks, on the comb path of bjj_verify_keyset_batch.  key_index[i] >= n_keys: that
 *     lane gets ok = 0, the other lanes are computed, and the call returns BJJ_ERR_ARG (a _dev call: the next bjj_sync).
 *   - _wide: any pk per lane, on bjj_verify_schnorr_batch's path after the reduction of s (off-curve pk or r replayed
 *     like there).
 *   The comb forms use h < Q raw against the key's table (never reduced mod SUBORDER), so keys with a torsion component
 *   give the reference's answer. */
int bjj_verify_schnorr_base_batch(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* msg32, const uint8_t* rx,
                                  const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok, uint8_t* status);
int bjj_verify_schnorr_base_batch_dev(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* msg32, const uint8_t* rx,
                                      const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok, uint8_t* status,
                                      void* stream);
int bjj_verify_schnorr_keyset_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index,
                                    const uint8_t* msg32, const uint8_t* rx, const uint8_t* ry, const uint8_t* s, int s_words,
                                    uint8_t* ok, uint8_t* status);
int bjj_verify_schnorr_keyset_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index,
                                        const uint8_t* msg32, const uint8_t* rx, const uint8_t* ry, const uint8_t* s,
                                        int s_words, uint8_t* ok, uint8_t* status, void* stream);
int bjj_verify_schnorr_wide_batch(bjj_ctx* ctx, size_t n, const uint8_t* pkx, const uint8_t* pky, const uint8_t* msg32,
                                  const uint8_t* rx, const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok,
                                  uint8_t* status);
int bjj_verify_schnorr_wide_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* pkx, const uint8_t* pky, const uint8_t* msg32,
                                      const uint8_t* rx, const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok,
                                      uint8_t* status, void* stream);

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
int bjj_multi_sign_schnorr_batch(bjj_multi* m, size_t n, const uint8_t* key32, const uint8_t* msg32, const uint8_t* nonce,
                                 int nonce_words, uint8_t* rx, uint8_t* ry, uint8_t* s, uint8_t* status);
int bjj_multi_fixed_base_batch(bjj_multi* m, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry);
int bjj_multi_decompress_batch(bjj_multi* m, size_t n, const uint8_t* in32, uint8_t* rx, uint8_t* ry, uint8_t* status);
/* bjj_msm_batch over the devices: each sums its shard of the points, and the N partial sums are summed by bjj_msm_batch
 * on device slot 0 with scalar 1 each (exact: the group sum).  Only those N points cross between devices, through the
 * host.  Errors and point_status as bjj_msm_batch. */
int bjj_multi_msm_batch(bjj_multi* m, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32, uint8_t* rx32,
                        uint8_t* ry32, uint8_t* point_status);

#ifdef __cplusplus
}
#endif
#endif /* BJJ_CUDA_H */
