// libbjj_cuda: kernels + C ABI (include/bjj_cuda.h).  sm_100a only; no CPU fallback.
//
// Kernel shape: one lane per thread, 128-thread CTAs, grid = min(ceil(n/128), SMs x resident CTAs)
// with a grid-stride loop, so every launch is a whole number of waves on the 148 SMs.  The work is
// bound by the integer-multiply (fma) pipe, not by HBM: a lane reads <= 192 B and executes ~10^5-10^6
// instructions.  Loads are two 16-byte vector loads per 32-byte element (1 KiB contiguous per warp).
#include <cuda_runtime.h>
#include <cudaTypedefs.h>   // PFN_cuMem*: the key-set tables' virtual memory calls, looked up at run time (libcuda is not linked)
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <new>
#include <random>
#include <utility>
#include <vector>

#include "../../include/bjj_cuda.h"
#include "kernels.h"
#include "msm.cuh"

using namespace bjj;

#define BJJ_PIPE_SLOTS 2

// integer environment knob (experiments and A/B runs; every default is the measured best)
static int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e && *e ? atoi(e) : dflt;
}
#define BJJ_CHUNK_LANES (1u << 20)
#define BJJ_CHUNK_RAMP_LANES ((size_t)1 << 18)   // first chunk of a long host call (see run_host)

// ---------------------------------------------------------------------------------------------------
// kernels
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(BJJ_BLOCK) k_comb_build(CombEntry* comb) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= BJJ_COMB_TOTAL) return;
    int w = (int)(idx / BJJ_COMB_ENTRIES), j = (int)(idx % BJJ_COMB_ENTRIES);
    comb_build_entry(comb, w, j);
}

// the table of the caller point (px, py) (bjj_base_create); thread 0 writes the BJJ_BASE_* outcome to *status
__global__ void __launch_bounds__(BJJ_BLOCK) k_comb_build_point(CombEntry* comb, const uint8_t* px, const uint8_t* py,
                                                                uint32_t* status) {
    size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= BJJ_COMB_TOTAL) return;
    const uint32_t st = lane_comb_build_point(comb, (int)(idx / BJJ_COMB_ENTRIES), (int)(idx % BJJ_COMB_ENTRIES), px, py);
    if (idx == 0) *status = st;
}

// key sets (bjj_keyset_create): check the keys and rewrite them in Montgomery form, then per sub-batch of keys the
// window chains (one thread per (key, window)) and the batched affine pass that writes the table entries
__global__ void __launch_bounds__(BJJ_BLOCK) k_keyset_check(size_t n, uint8_t* kx, uint8_t* ky, uint8_t* status) {
    BJJ_LANE_LOOP(n) status[i] = (uint8_t)lane_keyset_check(kx, ky, i);
}
__global__ void __launch_bounds__(BJJ_BLOCK) k_keyset_build(size_t keys, const uint8_t* kx, const uint8_t* ky, ProjScratch scr,
                                                            CombEntry* tables) {
    BJJ_LANE_LOOP(keys * Comb8::WINDOWS) {
        const size_t k = i / Comb8::WINDOWS;
        lane_keyset_build(kx, ky, k, (int)(i % Comb8::WINDOWS), scr, k * BJJ_KEY_BUILD_POINTS, tables + k * BJJ_KEY_COMB_TOTAL);
    }
}
__global__ void __launch_bounds__(BJJ_BLOCK) k_keyset_affine(size_t n, ProjScratch scr, CombEntry* tables) {
    batch_affine_strided(scr, KeysetCombOut{tables}, n, (size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x);
}

// s mod SUBORDER of the signer's wide s (nwords words per lane) into 32 B per lane (bjj_verify_schnorr_wide)
__global__ void __launch_bounds__(BJJ_BLOCK) k_mod_suborder_wide(size_t n, const uint8_t* wide, int nwords, uint8_t* out32) {
    BJJ_LANE_LOOP(n) {
        uint32_t acc[8];
        lane_mod_suborder_wide(acc, wide, nwords, i);
        store_u256(out32, i, acc);
    }
}

__global__ void __launch_bounds__(BJJ_BLOCK) k_split_scalars(size_t n, const uint8_t* h32, const uint8_t* s32, uint8_t* u32,
                                                             uint8_t* v32, uint8_t* w32) {
    BJJ_LANE_LOOP(n) lane_split_scalars(h32, s32, u32, v32, w32, i);
}

__global__ void __launch_bounds__(BJJ_BLOCK) k_fr_op(int op, size_t n, const uint8_t* a, const uint8_t* b,
                                                     uint8_t* out, uint32_t* gflags) {
    BJJ_FLAGS_BEGIN
    BJJ_LANE_LOOP(n) lane_fr_op(op, a, b, out, i, flags);
    BJJ_FLAGS_END(gflags)
}

__global__ void __launch_bounds__(BJJ_BLOCK) k_add(size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz,
                                                   const uint8_t* qx, const uint8_t* qy, const uint8_t* qz,
                                                   uint8_t* rx, uint8_t* ry, uint8_t* rz, uint32_t* gflags) {
    BJJ_FLAGS_BEGIN
    BJJ_LANE_LOOP(n) lane_add(px, py, pz, qx, qy, qz, rx, ry, rz, i, flags);
    BJJ_FLAGS_END(gflags)
}

__global__ void __launch_bounds__(BJJ_BLOCK) k_affine(size_t n, const uint8_t* px, const uint8_t* py,
                                                      const uint8_t* pz, uint8_t* rx, uint8_t* ry, uint32_t* gflags) {
    BJJ_FLAGS_BEGIN
    BJJ_LANE_LOOP(n) lane_affine(px, py, pz, rx, ry, i, flags);
    BJJ_FLAGS_END(gflags)
}

// projective scratch -> canonical affine outputs, one Fermat inversion per THREAD (Montgomery's trick)
__global__ void __launch_bounds__(BJJ_BLOCK) k_batch_affine(size_t n, ProjScratch scr, uint8_t* rx, uint8_t* ry) {
    batch_affine_strided(scr, rx, ry, n, (size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x);
}
// the same pass writing Point::compress of each affine result: one 32-byte plane instead of two
__global__ void __launch_bounds__(BJJ_BLOCK) k_batch_affine_compressed(size_t n, ProjScratch scr, uint8_t* out32) {
    batch_affine_strided(scr, CompressedOut{out32}, n, (size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x);
}

// The point kernels claim their lanes dynamically (BJJ_CLAIM_LOOP), like the verify kernels: with a static grid-stride
// split the kernel lasts as long as its slowest CTA and ncu showed 80 % (k_fixed_base, k_public) and 68 %
// (k_decompress_finish) of the resident warps active on average.  BJJ_POINT_CLAIM=0 restores the static split.
#ifndef BJJ_POINT_CLAIM
#define BJJ_POINT_CLAIM 1
#endif
#if BJJ_POINT_CLAIM
#define BJJ_POINT_LOOP(n, work) BJJ_CLAIM_LOOP(n, work) if (i < (n))
#else
#define BJJ_POINT_LOOP(n, work) BJJ_LANE_LOOP(n)
#endif
__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_fixed_base(size_t n, const uint8_t* k, ProjScratch scr,
                                                          const CombEntry* comb, unsigned long long* work) {
    BJJ_POINT_LOOP(n, work) lane_fixed_base(k, scr, i, comb);
}

__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_fixed_base2(size_t n, const uint8_t* k, const uint8_t* l, ProjScratch scr,
                                                           const CombEntry* comb_p, const CombEntry* comb_q,
                                                           unsigned long long* work) {
    BJJ_POINT_LOOP(n, work) lane_fixed_base2(k, l, scr, i, comb_p, comb_q);
}

// P_{key_index[i]}.mul_scalar(k) over a key set's compact tables (bjj_keyset_mul)
__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_keyset_mul(size_t n, const uint8_t* k, const uint8_t* key_index, uint32_t n_keys,
                                                          const CombEntry* tables, ProjScratch scr, uint32_t* gflags,
                                                          unsigned long long* work) {
    BJJ_FLAGS_BEGIN
    BJJ_POINT_LOOP(n, work) lane_keyset_mul(k, key_index, n_keys, tables, scr, i, flags);
    BJJ_FLAGS_END(gflags)
}

// the key of a key set whose compressed bytes are pk32[i], or BJJ_KEY_NONE (bjj_keyset_lookup)
__global__ void __launch_bounds__(BJJ_BLOCK) k_keyset_lookup(size_t n, const uint8_t* pk32, const uint8_t* comp, const uint32_t* slots,
                                                             uint64_t mask, uint64_t seed, uint32_t* key_index,
                                                             unsigned long long* work) {
    BJJ_POINT_LOOP(n, work) lane_keyset_lookup(pk32, comp, slots, mask, seed, key_index, i);
}

#ifndef BJJ_PUBLIC_BALLAST
#define BJJ_PUBLIC_BALLAST 1
#endif
__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_public(size_t n, const uint8_t* key, ProjScratch scr,
                                                      const CombEntry* comb, unsigned long long* work) {
    BJJ_POINT_LOOP(n, work) lane_public(key, scr, i, comb);
#if BJJ_PUBLIC_BALLAST
    fma_ballast(comb == nullptr, (uint32_t)n, scr.y);      // never taken (fr.cuh): BLAKE-512 makes this kernel ALU-heavy
#endif
}

__global__ void __launch_bounds__(BJJ_BLOCK) k_scalar_key(size_t n, const uint8_t* key, uint8_t* out) {
    BJJ_LANE_LOOP(n) lane_scalar_key(key, out, i);
}

__global__ void __launch_bounds__(BJJ_BLOCK) k_compress(size_t n, const uint8_t* px, const uint8_t* py, uint8_t* out,
                                                        uint32_t* gflags) {
    BJJ_FLAGS_BEGIN
    BJJ_LANE_LOOP(n) lane_compress(px, py, out, i, flags);
    BJJ_FLAGS_END(gflags)
}

// decompress_point in three phases around ONE shared inversion per thread (lanes.cuh): prepare (u, v) ->
// batched inverse of v -> square root + sign rule.  `slot0` offsets the scratch slots so that the R8 and A
// points of verify_compressed share one inversion pass.
__global__ void __launch_bounds__(BJJ_BLOCK) k_decompress_prepare(size_t n, const uint8_t* in, size_t stride, size_t off,
                                                                  ProjScratch scr, size_t slot0) {
    BJJ_LANE_LOOP(n) lane_decompress_prepare(in, stride, off, scr, slot0 + i, i);
}
__global__ void __launch_bounds__(BJJ_BLOCK) k_batch_inverse(size_t n, ProjScratch scr) {
    batch_inverse_strided(scr, n, (size_t)blockIdx.x * blockDim.x + threadIdx.x, (size_t)gridDim.x * blockDim.x);
}
__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_decompress_finish(size_t n, const uint8_t* in, size_t stride, size_t off,
                                                                 ProjScratch scr, size_t slot0, uint8_t* rx, uint8_t* ry,
                                                                 uint8_t* status, int merge, unsigned long long* work) {
    BJJ_POINT_LOOP(n, work) lane_decompress_finish(in, stride, off, scr, slot0 + i, rx, ry, status, i, merge != 0);
}

// ---------------------------------------------------------------------------------------------------
// context
// ---------------------------------------------------------------------------------------------------
// scratch that a launch needs besides its arguments: per-thread window tables and the exact-lane queue
struct Workspace {
    U128* table;
    size_t table_slots;
    uint32_t* exact_count;   // two device words (one per queue)
    uint32_t* exact_list;    // 2 x exact_cap indices
    size_t exact_cap;
    uint8_t* proj;           // 4 x 32 B per lane: X, Y, Z, running product
    size_t proj_lanes;
    uint8_t* vs;             // verify scratch: hm, u, v, w + decompressed R8, A (8 x 32 B per lane)
    size_t vs_lanes;
    uint8_t* kred;           // wide scalars reduced mod ORDER (32 B per lane)
    size_t kred_lanes;
    unsigned long long* claim;      // BJJ_CLAIM_SLOTS lane-claim counters of the point kernels, handed out round-robin
    unsigned claim_next;
    cudaStream_t aux;        // side stream: the exact-lane kernel overlaps the fast EC kernel
    cudaEvent_t ev_fork, ev_join;
};

// one of the two staging buffers of the host-pointer flavour: a copy stream, a device arena, and the events that
// order its copies against the (single) compute stream
struct PipeSlot {
    cudaStream_t stream;
    uint8_t* arena;
    size_t arena_bytes;
    cudaEvent_t ev_in, ev_out;
    // pageable caller arrays (what a plain Vec<u8> / malloc gives): page-locked mirror of the arena, same layout.  The
    // calling thread copies a chunk's inputs in while the GPU works on the chunk before, and copies a chunk's outputs
    // out ("drain") when the slot comes round again -- a cudaMemcpyAsync on pageable memory would block it instead.
    uint8_t* hstage;
    size_t hstage_bytes;
    cudaEvent_t ev_done;       // after the slot's device-to-host copies
    bool drain_pending;
    size_t drain_off, drain_lanes;
};

// scratch of bjj_msm_batch, grown on demand: per sub-batch of points the Niels entries and the pairs (two key and two
// value arrays of WINDOWS x points entries, the sort's double buffers) with the sort's temporary storage, the boundary
// lists of the accumulate levels (a uint32 key and a 128-byte point per slot, two ping-pong buffers); per call the
// buckets (WINDOWS x 2^(c-1) points of 128 B: 71 MB at c = 16), the segment and window sums, the flags word of the call
// and the 64-byte result of the host flavour
struct MsmWork {
    CombEntry* niels;
    size_t niels_cap;
    uint32_t* pairs;
    size_t pairs_cap;
    uint8_t* sort_temp;
    size_t sort_temp_cap;
    uint8_t* bound[2];
    size_t bound_cap[2];
    uint8_t* status;         // the point_status of a call that passes NULL
    size_t status_cap;
    uint8_t* sums;           // buckets, then segment results, then window sums, then the flags word and the result
    size_t sums_cap;
};

struct bjj_ctx {
    int device;
    int sms;
    cudaStream_t stream;        // stream of the _dev flavour when the caller passes NULL
    CombEntry* comb;
    Workspace ws;               // scratch of the kernels; all compute of a context runs on one stream at a time
    Workspace ws2;              // second set: the host flavour alternates, so a chunk's exact lanes may outlive it
    uint32_t* flags_dev;
    uint32_t* flags_host;       // pinned
    PipeSlot slot[BJJ_PIPE_SLOTS];
    unsigned long long launches;
    cudaError_t last;
    bool verify_split;          // half-size scalars in verify (split.cuh); BJJ_VERIFY_SPLIT=0 turns it off
    bool sign_fused;            // BJJ_SIGN_FUSED=1: sign as ONE kernel (k_sign) instead of the pipeline of launch_sign
    bool public_fused;          // BJJ_PUBLIC_FUSED=1: PrivateKey::public as ONE kernel (k_public) instead of k_scalar_key + k_fixed_base
    size_t lane_hint;           // host flavour: the largest chunk of the running call, so that lane-sized scratch is
                                // allocated ONCE up front (a cudaFree in mid-pipeline is a device-wide synchronisation)
    MsmWork msm;
};

// the comb table of a caller point, on the device of the context that built it, and the point's canonical affine
// coordinates (little-endian bytes; verify_base hashes them)
struct bjj_base {
    bjj_ctx* ctx;
    CombEntry* comb;
    uint8_t x[32], y[32];
};

// N keys with their compact combs (bjj_keyset_create), on the device of the context that built them: `keys` holds the
// x plane then the y plane (Montgomery form, 32 B per key each), `tables` the N Comb8 tables.  `index` is the lookup by
// compressed bytes (lanes.cuh: keyset_index_build): compress(P_j) (32 B per key), then `slot_mask` + 1 uint32 slots,
// then one flags word that the lookup verify passes to its kernels instead of the context's (nobody reads it).
// The tables grow in place (bjj_keyset_append): `tables` is the start of a reserved virtual range of `va_bytes`, room
// for the most keys the device's memory could hold, of which the first `mapped` bytes (a multiple of `gran`) are backed
// by the physical allocations `maps` (offset, bytes), one per call that grew the set.  `comp` is a host copy of the
// compressed keys, from which an edit rebuilds the slots.
struct bjj_keyset {
    bjj_ctx* ctx = nullptr;
    size_t n_keys = 0;
    uint8_t* keys = nullptr;
    CombEntry* tables = nullptr;
    uint8_t* index = nullptr;
    uint64_t slot_mask = 0;
    uint64_t seed = 0;
    size_t va_bytes = 0, mapped = 0, gran = 0;
    std::vector<std::pair<size_t, size_t>> maps;
    std::vector<uint8_t> comp;
};

static const uint8_t* keyset_comp(const bjj_keyset* ks) { return ks->index; }
static const uint32_t* keyset_slots(const bjj_keyset* ks) { return (const uint32_t*)(ks->index + 32 * ks->n_keys); }
static uint32_t* keyset_quiet_flags(const bjj_keyset* ks) { return (uint32_t*)(ks->index + 32 * ks->n_keys) + ks->slot_mask + 1; }
// a key-set call names its set: NULL or a handle of another context is an argument error
static bool keyset_of(bjj_ctx* ctx, const bjj_keyset* ks) { return ks && ks->ctx == ctx; }

#define CU(ctx, call)                      \
    do {                                   \
        cudaError_t e_ = (call);           \
        if (e_ != cudaSuccess) {           \
            (ctx)->last = e_;              \
            return BJJ_ERR_CUDA;           \
        }                                  \
    } while (0)

// propagates a nonzero BJJ_ERR_* code
#define TRY(call)                \
    do {                         \
        int rc_ = (call);        \
        if (rc_) return rc_;     \
    } while (0)

// counts `count` kernel launches (bjj_kernel_launches) and reports a failed launch among them
static int launched(bjj_ctx* ctx, int count = 1) {
    ctx->launches += count;
    CU(ctx, cudaGetLastError());
    return BJJ_OK;
}

static int grid_cap(bjj_ctx* ctx, int per_sm, size_t n) {
    size_t want = (n + BJJ_BLOCK - 1) / BJJ_BLOCK;
    size_t cap = (size_t)ctx->sms * (per_sm < 1 ? 1 : per_sm);
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

template <class Kernel>
static int grid_for(bjj_ctx* ctx, Kernel* kernel, size_t n) {
    return grid_cap(ctx, bjjk::blocks_per_sm(kernel), n);
}

// Grow-only scratch: afterwards *buf holds at least `want` units of `unit` bytes.  It is reallocated, contents lost,
// only when it held fewer; the old buffer is freed first so that the two never coexist.  `pinned`: page-locked host
// memory instead of device memory.
template <class T>
static int grow(bjj_ctx* ctx, T** buf, size_t* cap, size_t want, size_t unit, bool pinned = false) {
    if (*cap >= want) return BJJ_OK;
    if (*buf) pinned ? cudaFreeHost(*buf) : cudaFree(*buf);
    *buf = nullptr;
    *cap = 0;
    CU(ctx, pinned ? cudaHostAlloc(buf, want * unit, cudaHostAllocDefault) : cudaMalloc(buf, want * unit));
    *cap = want;
    return BJJ_OK;
}

// sub-batch size of the point kernels: bounds the projective scratch at 4 x 32 B x 2^21 = 256 MiB
#define BJJ_POINT_SUBBATCH ((size_t)1 << 21)

// Lanes that the lane-sized scratch of a workspace must hold for a call of n lanes: one sub-batch, and at least the
// host flavour's largest chunk (lane_hint), so that a long host call allocates once up front.
static size_t scratch_lanes(bjj_ctx* ctx, size_t n) {
    const size_t lanes = n < BJJ_POINT_SUBBATCH ? n : BJJ_POINT_SUBBATCH;
    return lanes < ctx->lane_hint ? ctx->lane_hint : lanes;
}

// f(off, m) on consecutive sub-batches [off, off + m) of at most BJJ_POINT_SUBBATCH lanes; stops at the first error
template <class F>
static int for_each_subbatch(size_t n, F f) {
    for (size_t off = 0; off < n; off += BJJ_POINT_SUBBATCH)
        TRY(f(off, n - off < BJJ_POINT_SUBBATCH ? n - off : BJJ_POINT_SUBBATCH));
    return BJJ_OK;
}

static int ensure_table(bjj_ctx* ctx, Workspace* ws, size_t slots) {
    return grow(ctx, &ws->table, &ws->table_slots, slots, BJJ_TABLE_U128_PER_LANE * sizeof(U128));
}

// makes room for two queues of `lanes` lane indices each and zeroes both counters on `st`
static int ensure_queue(bjj_ctx* ctx, Workspace* ws, size_t lanes, cudaStream_t st, ExactQueue* q, ExactQueue* q2 = nullptr) {
    // 48 bytes: the two queue counters, then (at byte 16) the lane-claim counters of the verify kernels (hash, Straus)
    // and (at byte 32) the claim counter of the exact-lane kernels
    if (!ws->exact_count) CU(ctx, cudaMalloc(&ws->exact_count, 48));
    TRY(grow(ctx, &ws->exact_list, &ws->exact_cap, lanes, 2 * sizeof(uint32_t)));
    CU(ctx, cudaMemsetAsync(ws->exact_count, 0, 48, st));
    q->count = ws->exact_count;
    q->list = ws->exact_list;
    if (q2) {
        q2->count = ws->exact_count + 1;
        q2->list = ws->exact_list + ws->exact_cap;
    }
    return BJJ_OK;
}

// A zeroed lane-claim counter for ONE launch on `st` (kernels.h::BJJ_CLAIM_LOOP).  Slots rotate, so that the memset of
// the next launch never touches the counter of a launch that is still running on the same stream order.
#define BJJ_CLAIM_SLOTS 16
static int claim_counter(bjj_ctx* ctx, Workspace* ws, cudaStream_t st, unsigned long long** out) {
    if (!ws->claim) CU(ctx, cudaMalloc(&ws->claim, BJJ_CLAIM_SLOTS * sizeof(unsigned long long)));
    unsigned long long* c = ws->claim + (ws->claim_next++ % BJJ_CLAIM_SLOTS);
    CU(ctx, cudaMemsetAsync(c, 0, sizeof(unsigned long long), st));
    *out = c;
    return BJJ_OK;
}

static unsigned long long* work_counters(Workspace* ws) { return reinterpret_cast<unsigned long long*>(ws->exact_count + 4); }

static int ensure_proj(bjj_ctx* ctx, Workspace* ws, size_t lanes, ProjScratch* scr) {
    TRY(grow(ctx, &ws->proj, &ws->proj_lanes, lanes, 128));
    scr->x = ws->proj;
    scr->y = scr->x + 32 * ws->proj_lanes;
    scr->z = scr->y + 32 * ws->proj_lanes;
    scr->p = scr->z + 32 * ws->proj_lanes;
    return BJJ_OK;
}

// grid of the batched affine pass: every thread should own >= 32 lanes so its one Fermat inversion
// (~380 fmul) is amortised, but never more threads than the device holds at once
static int affine_grid(bjj_ctx* ctx, size_t n) {
    size_t want = (n / 32 + BJJ_BLOCK - 1) / BJJ_BLOCK;
    size_t cap = (size_t)ctx->sms * 8;
    if (want < 1) want = 1;
    return (int)(want < cap ? want : cap);
}

static int ensure_aux(bjj_ctx* ctx, Workspace* ws) {
    if (ws->aux) return BJJ_OK;
    CU(ctx, cudaStreamCreateWithFlags(&ws->aux, cudaStreamNonBlocking));
    CU(ctx, cudaEventCreateWithFlags(&ws->ev_fork, cudaEventDisableTiming));
    CU(ctx, cudaEventCreateWithFlags(&ws->ev_join, cudaEventDisableTiming));
    return BJJ_OK;
}

static void free_workspace(Workspace* ws) {
    if (ws->aux) {
        cudaStreamSynchronize(ws->aux);
        cudaEventDestroy(ws->ev_fork);
        cudaEventDestroy(ws->ev_join);
        cudaStreamDestroy(ws->aux);
    }
    if (ws->table) cudaFree(ws->table);
    if (ws->proj) cudaFree(ws->proj);
    if (ws->vs) cudaFree(ws->vs);
    if (ws->kred) cudaFree(ws->kred);
    if (ws->exact_count) cudaFree(ws->exact_count);
    if (ws->claim) cudaFree(ws->claim);
    if (ws->exact_list) cudaFree(ws->exact_list);
    memset(ws, 0, sizeof(*ws));
}

extern "C" {

int bjj_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) return 0;
    return n;
}

const char* bjj_error_string(int code) {
    switch (code) {
        case BJJ_OK: return "ok";
        case BJJ_ERR_CUDA: return "CUDA runtime error";
        case BJJ_ERR_ARG: return "invalid argument";
        case BJJ_ERR_NONCANONICAL: return "field element input >= Q (results computed mod Q)";
        case BJJ_ERR_NOMEM: return "out of memory";
        default: return "unknown error";
    }
}

const char* bjj_status_string(int status) {
    switch (status) {
        case BJJ_STATUS_OK: return "";
        case BJJ_STATUS_Y_RANGE: return "y outside the Finite Field over R";
        case BJJ_STATUS_NO_INV: return "no mod inv of Zero";
        case BJJ_STATUS_NOT_SQUARE: return "not a mod p square";
        case BJJ_STATUS_MSG_RANGE: return "msg outside the Finite Field";
        default: return "unknown status";
    }
}

const char* bjj_last_cuda_error(bjj_ctx* ctx) { return ctx ? cudaGetErrorString(ctx->last) : "no context"; }
void* bjj_stream(bjj_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int bjj_device(bjj_ctx* ctx) { return ctx ? ctx->device : -1; }
unsigned long long bjj_kernel_launches(bjj_ctx* ctx) { return ctx ? ctx->launches : 0; }

void* bjj_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
void bjj_host_free(void* p) {
    if (p) cudaFreeHost(p);
}
void* bjj_dev_alloc(bjj_ctx* ctx, size_t bytes) {
    if (!ctx) return nullptr;
    void* p = nullptr;
    cudaSetDevice(ctx->device);
    if (cudaMalloc(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}
void bjj_dev_free(bjj_ctx* ctx, void* p) {
    if (!ctx || !p) return;
    cudaSetDevice(ctx->device);
    cudaFree(p);
}
int bjj_memcpy_h2d(bjj_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (!ctx) return BJJ_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, ctx->stream));
    return BJJ_OK;
}
int bjj_memcpy_d2h(bjj_ctx* ctx, void* dst, const void* src, size_t bytes) {
    if (!ctx) return BJJ_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    return BJJ_OK;
}

void bjj_destroy(bjj_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (int s = 0; s < BJJ_PIPE_SLOTS; s++) {
        if (ctx->slot[s].arena) cudaFree(ctx->slot[s].arena);
        if (ctx->slot[s].hstage) cudaFreeHost(ctx->slot[s].hstage);
        if (ctx->slot[s].ev_done) cudaEventDestroy(ctx->slot[s].ev_done);
        if (ctx->slot[s].ev_in) cudaEventDestroy(ctx->slot[s].ev_in);
        if (ctx->slot[s].ev_out) cudaEventDestroy(ctx->slot[s].ev_out);
        if (ctx->slot[s].stream) cudaStreamDestroy(ctx->slot[s].stream);
    }
    free_workspace(&ctx->ws);
    free_workspace(&ctx->ws2);
    for (void* p : {(void*)ctx->msm.niels, (void*)ctx->msm.pairs, (void*)ctx->msm.sort_temp, (void*)ctx->msm.bound[0],
                    (void*)ctx->msm.bound[1], (void*)ctx->msm.status, (void*)ctx->msm.sums})
        if (p) cudaFree(p);
    if (ctx->comb) cudaFree(ctx->comb);
    if (ctx->flags_dev) cudaFree(ctx->flags_dev);
    if (ctx->flags_host) cudaFreeHost(ctx->flags_host);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    free(ctx);
}

int bjj_init(int device, bjj_ctx** out) {
    if (!out) return BJJ_ERR_ARG;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || device < 0 || device >= count) return BJJ_ERR_CUDA;
    bjj_ctx* ctx = (bjj_ctx*)calloc(1, sizeof(bjj_ctx));
    if (!ctx) return BJJ_ERR_NOMEM;
    ctx->device = device;
    ctx->last = cudaSuccess;
    {
        const char* e = getenv("BJJ_VERIFY_SPLIT");
        ctx->verify_split = !(e && e[0] == '0');
        e = getenv("BJJ_SIGN_FUSED");
        ctx->sign_fused = e && e[0] == '1';
        e = getenv("BJJ_PUBLIC_FUSED");
        ctx->public_fused = e && e[0] == '1';
    }
#define INIT_CU(call)                  \
    do {                               \
        cudaError_t e_ = (call);       \
        if (e_ != cudaSuccess) {       \
            fprintf(stderr, "libbjj_cuda: %s failed: %s\n", #call, cudaGetErrorString(e_)); \
            bjj_destroy(ctx);          \
            return BJJ_ERR_CUDA;       \
        }                              \
    } while (0)
    INIT_CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    INIT_CU(cudaGetDeviceProperties(&prop, device));
    ctx->sms = prop.multiProcessorCount;
    INIT_CU(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    for (int s = 0; s < BJJ_PIPE_SLOTS; s++) {
        INIT_CU(cudaStreamCreateWithFlags(&ctx->slot[s].stream, cudaStreamNonBlocking));
        INIT_CU(cudaEventCreateWithFlags(&ctx->slot[s].ev_in, cudaEventDisableTiming));
        INIT_CU(cudaEventCreateWithFlags(&ctx->slot[s].ev_out, cudaEventDisableTiming));
        INIT_CU(cudaEventCreateWithFlags(&ctx->slot[s].ev_done, cudaEventDisableTiming));
    }
    INIT_CU(cudaMalloc(&ctx->flags_dev, sizeof(uint32_t)));
    INIT_CU(cudaMemsetAsync(ctx->flags_dev, 0, sizeof(uint32_t), ctx->stream));
    INIT_CU(cudaHostAlloc(&ctx->flags_host, sizeof(uint32_t), cudaHostAllocDefault));
    const size_t comb_bytes = BJJ_COMB_TOTAL * sizeof(CombEntry);
    INIT_CU(cudaMalloc(&ctx->comb, comb_bytes));
    INIT_CU(cudaMemsetAsync(ctx->comb, 0, comb_bytes, ctx->stream));
    const size_t total = BJJ_COMB_TOTAL;
    k_comb_build<<<(total + BJJ_BLOCK - 1) / BJJ_BLOCK, BJJ_BLOCK, 0, ctx->stream>>>(ctx->comb);
    ctx->launches++;
    INIT_CU(cudaGetLastError());
    INIT_CU(cudaStreamSynchronize(ctx->stream));
#undef INIT_CU
    *out = ctx;
    return BJJ_OK;
}

// waits for the ctx stream and all pipeline slots; returns + clears the sticky error flags
int bjj_sync(bjj_ctx* ctx) {
    if (!ctx) return BJJ_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    for (int s = 0; s < BJJ_PIPE_SLOTS; s++) CU(ctx, cudaStreamSynchronize(ctx->slot[s].stream));
    CU(ctx, cudaMemcpyAsync(ctx->flags_host, ctx->flags_dev, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaMemsetAsync(ctx->flags_dev, 0, sizeof(uint32_t), ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    uint32_t f = *ctx->flags_host;
    if (f & (BJJ_FLAG_KEY_INDEX | BJJ_FLAG_OFF_CURVE)) return BJJ_ERR_ARG;
    if (f & BJJ_FLAG_NONCANONICAL) return BJJ_ERR_NONCANONICAL;
    return BJJ_OK;
}

}  // extern "C"

// builds the table of (px32, py32) into a new *comb and leaves the BJJ_BASE_* outcome in *status; `io` is device
// scratch of 80 bytes (the point in, the outcome out)
static int build_base_comb(bjj_ctx* ctx, const uint8_t* px32, const uint8_t* py32, uint8_t* io, CombEntry** comb,
                           uint32_t* status) {
    CU(ctx, cudaMalloc(comb, BJJ_COMB_TOTAL * sizeof(CombEntry)));
    CU(ctx, cudaMemcpyAsync(io, px32, 32, cudaMemcpyHostToDevice, ctx->stream));
    CU(ctx, cudaMemcpyAsync(io + 32, py32, 32, cudaMemcpyHostToDevice, ctx->stream));
    const size_t total = BJJ_COMB_TOTAL;
    k_comb_build_point<<<(total + BJJ_BLOCK - 1) / BJJ_BLOCK, BJJ_BLOCK, 0, ctx->stream>>>(*comb, io, io + 32, (uint32_t*)(io + 64));
    TRY(launched(ctx));
    CU(ctx, cudaMemcpyAsync(status, io + 64, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return BJJ_OK;
}

// the table that `base` names for a call on ctx: B8's for NULL, nullptr for a handle of another context
static const CombEntry* base_comb(bjj_ctx* ctx, const bjj_base* base) {
    if (!base) return ctx->comb;
    return base->ctx == ctx ? base->comb : nullptr;
}

extern "C" {

int bjj_base_create(bjj_ctx* ctx, const uint8_t* px32, const uint8_t* py32, bjj_base** out) {
    if (!out) return BJJ_ERR_ARG;
    *out = nullptr;
    if (!ctx || !px32 || !py32) return BJJ_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    uint8_t* io = nullptr;
    CU(ctx, cudaMalloc(&io, 80));
    CombEntry* comb = nullptr;
    uint32_t status = BJJ_BASE_OK;
    int rc = build_base_comb(ctx, px32, py32, io, &comb, &status);
    cudaFree(io);
    if (rc == BJJ_OK && status != BJJ_BASE_OK) rc = status == BJJ_BASE_NONCANONICAL ? BJJ_ERR_NONCANONICAL : BJJ_ERR_ARG;
    bjj_base* b = rc == BJJ_OK ? (bjj_base*)malloc(sizeof(bjj_base)) : nullptr;
    if (rc == BJJ_OK && !b) rc = BJJ_ERR_NOMEM;
    if (rc != BJJ_OK) {
        if (comb) cudaFree(comb);
        return rc;
    }
    b->ctx = ctx;
    b->comb = comb;
    memcpy(b->x, px32, 32);
    memcpy(b->y, py32, 32);
    *out = b;
    return BJJ_OK;
}

void bjj_base_destroy(bjj_ctx* ctx, bjj_base* base) {
    if (!ctx || !base || base->ctx != ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();      // calls on any stream may still read the table
    cudaFree(base->comb);
    free(base);
}

// keys per build sub-batch of the key-set build: their build lanes fit the point kernels' sub-batch of scratch
#define BJJ_KEYSET_SUBBATCH (BJJ_POINT_SUBBATCH / BJJ_KEY_BUILD_POINTS)
#define BJJ_KEY_TABLE_BYTES ((size_t)BJJ_KEY_COMB_TOTAL * sizeof(CombEntry))

// cudaMalloc that reports a failure as BJJ_ERR_NOMEM with the CUDA error cleared: the tables of a large key set may
// simply not fit
static int dev_alloc(void** p, size_t bytes) {
    if (cudaMalloc(p, bytes) == cudaSuccess) return BJJ_OK;
    cudaGetLastError();
    *p = nullptr;
    return BJJ_ERR_NOMEM;
}

// The driver's virtual memory management, resolved once through the runtime so that libbjj_cuda.so loads where there
// is no driver.  `ok` is false when an entry point is missing.
struct VmmApi {
    PFN_cuMemGetAllocationGranularity granularity;
    PFN_cuMemAddressReserve reserve;
    PFN_cuMemAddressFree address_free;
    PFN_cuMemCreate create;
    PFN_cuMemRelease release;
    PFN_cuMemMap map;
    PFN_cuMemUnmap unmap;
    PFN_cuMemSetAccess set_access;
    bool ok;
};
static const VmmApi& vmm() {
    static const VmmApi api = [] {
        VmmApi a{};
        auto get = [](const char* name, auto* fn) {
            cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
            return cudaGetDriverEntryPoint(name, (void**)fn, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess;
        };
        a.ok = get("cuMemGetAllocationGranularity", &a.granularity) && get("cuMemAddressReserve", &a.reserve) &&
               get("cuMemAddressFree", &a.address_free) && get("cuMemCreate", &a.create) && get("cuMemRelease", &a.release) &&
               get("cuMemMap", &a.map) && get("cuMemUnmap", &a.unmap) && get("cuMemSetAccess", &a.set_access);
        cudaGetLastError();
        return a;
    }();
    return api;
}

static CUmemAllocationProp device_alloc_prop(int device) {
    CUmemAllocationProp prop = {};
    prop.type = CU_MEM_ALLOCATION_TYPE_PINNED;
    prop.location.type = CU_MEM_LOCATION_TYPE_DEVICE;
    prop.location.id = device;
    return prop;
}

// reserves ks's table range: (total device memory / 396,480 B) tables, rounded up to the allocation granularity.  No
// set can hold more keys, so the range never has to move.
static int tables_reserve(bjj_ctx* ctx, bjj_keyset* ks) {
    const VmmApi& v = vmm();
    if (!v.ok) {
        ctx->last = cudaErrorNotSupported;
        return BJJ_ERR_CUDA;
    }
    size_t free_b = 0, total_b = 0;
    CU(ctx, cudaMemGetInfo(&free_b, &total_b));
    const CUmemAllocationProp prop = device_alloc_prop(ctx->device);
    if (v.granularity(&ks->gran, &prop, CU_MEM_ALLOC_GRANULARITY_MINIMUM) != CUDA_SUCCESS || !ks->gran) return BJJ_ERR_NOMEM;
    const size_t bytes = total_b / BJJ_KEY_TABLE_BYTES * BJJ_KEY_TABLE_BYTES;
    ks->va_bytes = (bytes + ks->gran - 1) / ks->gran * ks->gran;
    CUdeviceptr va = 0;
    if (v.reserve(&va, ks->va_bytes, 0, 0, 0) != CUDA_SUCCESS) {
        ks->va_bytes = 0;
        return BJJ_ERR_NOMEM;
    }
    ks->tables = (CombEntry*)va;
    return BJJ_OK;
}

// unmaps the physical allocations maps[from..] (their memory is freed with the mapping: each handle was released once
// mapped)
static void tables_unmap_from(bjj_keyset* ks, size_t from) {
    while (ks->maps.size() > from) {
        const std::pair<size_t, size_t> m = ks->maps.back();
        vmm().unmap((CUdeviceptr)ks->tables + m.first, m.second);
        ks->mapped = m.first;
        ks->maps.pop_back();
    }
}

// backs the tables of n keys with physical memory: one more allocation after the mapped part (whose last granule the
// previous keys may fill only partly).  Anything but success leaves the mapping as it was and returns BJJ_ERR_NOMEM.
static int tables_grow(bjj_ctx* ctx, bjj_keyset* ks, size_t n) {
    const VmmApi& v = vmm();
    if (n > ks->va_bytes / BJJ_KEY_TABLE_BYTES) return BJJ_ERR_NOMEM;
    const size_t need = (n * BJJ_KEY_TABLE_BYTES + ks->gran - 1) / ks->gran * ks->gran;
    if (need <= ks->mapped) return BJJ_OK;
    const size_t off = ks->mapped, bytes = need - off;
    const CUdeviceptr at = (CUdeviceptr)ks->tables + off;
    const CUmemAllocationProp prop = device_alloc_prop(ctx->device);
    CUmemGenericAllocationHandle h;
    if (v.create(&h, bytes, &prop, 0) != CUDA_SUCCESS) return BJJ_ERR_NOMEM;
    const bool mapped = v.map(at, bytes, 0, h, 0) == CUDA_SUCCESS;
    v.release(h);
    if (!mapped) return BJJ_ERR_NOMEM;
    CUmemAccessDesc acc = {};
    acc.location = prop.location;
    acc.flags = CU_MEM_ACCESS_FLAGS_PROT_READWRITE;
    ks->maps.push_back({off, bytes});
    ks->mapped = need;
    if (v.set_access(at, bytes, &acc, 1) != CUDA_SUCCESS) {
        tables_unmap_from(ks, ks->maps.size() - 1);
        return BJJ_ERR_NOMEM;
    }
    return BJJ_OK;
}

static void keyset_free(bjj_keyset* ks) {
    if (ks->keys) cudaFree(ks->keys);
    if (ks->index) cudaFree(ks->index);
    if (ks->tables) {
        tables_unmap_from(ks, 0);
        vmm().address_free((CUdeviceptr)ks->tables, ks->va_bytes);
    }
    delete ks;
}

// uploads n keys (canonical SoA ax, ay) into `stage` (x plane, y plane, one status byte per key: 65 B per key), checks
// them and rewrites them in Montgomery form (k_keyset_check, one launch).  key_status (may be NULL) receives one
// BJJ_KEY_* code per key.  A coordinate >= Q outranks a key off the curve; the reference's product with an off-curve
// key depends on its double-and-add order, which a comb does not follow, so such keys are refused as by bjj_base_create.
static int keyset_check(bjj_ctx* ctx, size_t n, const uint8_t* ax, const uint8_t* ay, uint8_t* stage, uint8_t* key_status) {
    uint8_t *kx = stage, *ky = kx + 32 * n, *st_dev = ky + 32 * n;
    cudaStream_t st = ctx->stream;
    uint8_t* status = (uint8_t*)malloc(n);
    if (!status) return BJJ_ERR_NOMEM;
    auto body = [&]() -> int {
        CU(ctx, cudaMemcpyAsync(kx, ax, 32 * n, cudaMemcpyHostToDevice, st));
        CU(ctx, cudaMemcpyAsync(ky, ay, 32 * n, cudaMemcpyHostToDevice, st));
        k_keyset_check<<<grid_for(ctx, k_keyset_check, n), BJJ_BLOCK, 0, st>>>(n, kx, ky, st_dev);
        TRY(launched(ctx));
        CU(ctx, cudaMemcpyAsync(status, st_dev, n, cudaMemcpyDeviceToHost, st));
        CU(ctx, cudaStreamSynchronize(st));
        if (key_status) memcpy(key_status, status, n);
        bool off = false;
        for (size_t j = 0; j < n; j++) {
            if (status[j] == BJJ_BASE_NONCANONICAL) return BJJ_ERR_NONCANONICAL;
            off = off || status[j] != BJJ_BASE_OK;
        }
        return off ? BJJ_ERR_ARG : BJJ_OK;
    };
    const int rc = body();
    free(status);
    return rc;
}

// the comb tables of n keys (Montgomery planes kx, ky, 32 B per key) into tables, key after key: per sub-batch of
// BJJ_KEYSET_SUBBATCH keys the window chains, then the batched affine pass (2 launches).  The build borrows the
// context's projective scratch, so the caller has synchronised the device (and grown the scratch: keyset_edit).
static int keyset_build_tables(bjj_ctx* ctx, size_t n, const uint8_t* kx, const uint8_t* ky, CombEntry* tables) {
    cudaStream_t st = ctx->stream;
    for (size_t k0 = 0; k0 < n; k0 += BJJ_KEYSET_SUBBATCH) {
        const size_t keys = n - k0 < BJJ_KEYSET_SUBBATCH ? n - k0 : BJJ_KEYSET_SUBBATCH;
        const size_t lanes = keys * BJJ_KEY_BUILD_POINTS;
        ProjScratch scr;
        TRY(ensure_proj(ctx, &ctx->ws, lanes, &scr));
        CombEntry* tbl = tables + k0 * BJJ_KEY_COMB_TOTAL;
        k_keyset_build<<<grid_for(ctx, k_keyset_build, keys * Comb8::WINDOWS), BJJ_BLOCK, 0, st>>>(keys, kx + 32 * k0, ky + 32 * k0,
                                                                                                 scr, tbl);
        k_keyset_affine<<<affine_grid(ctx, lanes), BJJ_BLOCK, 0, st>>>(lanes, scr, tbl);
        TRY(launched(ctx, 2));
    }
    return BJJ_OK;
}

// keys first .. first + n - 1 of ks get the coordinates ax, ay (first == ks->n_keys appends them): create, append and
// replace all come here.  Everything the edit allocates comes first and every check passes before the set changes; on
// an error before that point the allocations are undone and the set is as it was.
static int keyset_edit(bjj_ctx* ctx, bjj_keyset* ks, size_t first, size_t n, const uint8_t* ax, const uint8_t* ay,
                       uint8_t* key_status) {
    CU(ctx, cudaSetDevice(ctx->device));
    // _dev calls on other streams may still read the planes, tables and index that this call changes or frees
    CU(ctx, cudaDeviceSynchronize());
    const size_t n0 = ks->n_keys, n1 = first + n > n0 ? first + n : n0;
    const size_t maps0 = ks->maps.size();
    cudaStream_t st = ctx->stream;
    uint8_t *stage = nullptr, *keys = ks->keys, *index = nullptr;
    std::vector<uint8_t> comp;
    uint64_t slot_mask = 0;
    auto body = [&]() -> int {
        TRY(dev_alloc((void**)&stage, 65 * n));
        TRY(keyset_check(ctx, n, ax, ay, stage, key_status));
        // the index of the edited key list, rebuilt on the host from the compressed keys
        comp.resize(32 * n1);
        if (n0) memcpy(comp.data(), ks->comp.data(), 32 * n0);
        for (size_t j = 0; j < n; j++) keyset_compress(ax, ay, j, comp.data() + 32 * (first + j));
        const size_t slots = keyset_index_slots(n1), index_bytes = 32 * n1 + 4 * slots + 4;
        std::vector<uint8_t> host_index(index_bytes, 0);
        memcpy(host_index.data(), comp.data(), 32 * n1);
        keyset_index_fill(n1, comp.data(), ks->seed, (uint32_t*)(host_index.data() + 32 * n1));
        slot_mask = slots - 1;
        TRY(dev_alloc((void**)&index, index_bytes));
        if (n1 > n0) {
            TRY(dev_alloc((void**)&keys, 64 * n1));
            TRY(tables_grow(ctx, ks, n1));
        }
        // the build's projective scratch, grown here so that nothing after this point allocates
        ProjScratch scr;
        const int rc_scr = ensure_proj(ctx, &ctx->ws, (n < BJJ_KEYSET_SUBBATCH ? n : BJJ_KEYSET_SUBBATCH) * BJJ_KEY_BUILD_POINTS, &scr);
        if (rc_scr != BJJ_OK) {
            if (ctx->last != cudaErrorMemoryAllocation) return rc_scr;
            cudaGetLastError();
            return BJJ_ERR_NOMEM;
        }
        // from here on the set changes
        uint8_t *kx = keys, *ky = keys + 32 * n1;
        if (keys != ks->keys && n0) {
            CU(ctx, cudaMemcpyAsync(kx, ks->keys, 32 * n0, cudaMemcpyDeviceToDevice, st));
            CU(ctx, cudaMemcpyAsync(ky, ks->keys + 32 * n0, 32 * n0, cudaMemcpyDeviceToDevice, st));
        }
        CU(ctx, cudaMemcpyAsync(kx + 32 * first, stage, 32 * n, cudaMemcpyDeviceToDevice, st));
        CU(ctx, cudaMemcpyAsync(ky + 32 * first, stage + 32 * n, 32 * n, cudaMemcpyDeviceToDevice, st));
        CU(ctx, cudaMemcpyAsync(index, host_index.data(), index_bytes, cudaMemcpyHostToDevice, st));
        TRY(keyset_build_tables(ctx, n, kx + 32 * first, ky + 32 * first, ks->tables + first * BJJ_KEY_COMB_TOTAL));
        CU(ctx, cudaStreamSynchronize(st));
        return BJJ_OK;
    };
    int rc;
    try {
        rc = body();
    } catch (const std::bad_alloc&) {
        rc = BJJ_ERR_NOMEM;
    }
    if (stage) cudaFree(stage);
    if (rc != BJJ_OK) {
        if (index) cudaFree(index);
        if (keys != ks->keys) cudaFree(keys);
        tables_unmap_from(ks, maps0);
        return rc;
    }
    if (keys != ks->keys && ks->keys) cudaFree(ks->keys);
    if (ks->index) cudaFree(ks->index);
    ks->keys = keys;
    ks->index = index;
    ks->slot_mask = slot_mask;
    ks->comp.swap(comp);
    ks->n_keys = n1;
    return BJJ_OK;
}

int bjj_keyset_create(bjj_ctx* ctx, size_t n_keys, const uint8_t* ax, const uint8_t* ay, uint8_t* key_status, bjj_keyset** out) {
    if (!out) return BJJ_ERR_ARG;
    *out = nullptr;
    if (!ctx || !ax || !ay || n_keys == 0 || n_keys > 0xFFFFFFFFull) return BJJ_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    bjj_keyset* ks = new (std::nothrow) bjj_keyset();
    if (!ks) return BJJ_ERR_NOMEM;
    ks->ctx = ctx;
    ks->seed = (uint64_t)std::random_device{}() << 32 ^ std::random_device{}();
    int rc = tables_reserve(ctx, ks);
    if (rc == BJJ_OK) rc = keyset_edit(ctx, ks, 0, n_keys, ax, ay, key_status);
    if (rc != BJJ_OK) {
        keyset_free(ks);
        return rc;
    }
    *out = ks;
    return BJJ_OK;
}

int bjj_keyset_append(bjj_ctx* ctx, bjj_keyset* ks, size_t n_new, const uint8_t* ax, const uint8_t* ay, uint8_t* key_status) {
    if (!keyset_of(ctx, ks) || n_new > 0xFFFFFFFFull - ks->n_keys) return BJJ_ERR_ARG;
    if (n_new == 0) return BJJ_OK;
    if (!ax || !ay) return BJJ_ERR_ARG;
    return keyset_edit(ctx, ks, ks->n_keys, n_new, ax, ay, key_status);
}

int bjj_keyset_replace(bjj_ctx* ctx, bjj_keyset* ks, size_t first, size_t count, const uint8_t* ax, const uint8_t* ay,
                       uint8_t* key_status) {
    if (!keyset_of(ctx, ks) || first > ks->n_keys || count > ks->n_keys - first) return BJJ_ERR_ARG;
    if (count == 0) return BJJ_OK;
    if (!ax || !ay) return BJJ_ERR_ARG;
    return keyset_edit(ctx, ks, first, count, ax, ay, key_status);
}

void bjj_keyset_destroy(bjj_ctx* ctx, bjj_keyset* ks) {
    if (!ctx || !ks || ks->ctx != ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();      // calls on any stream may still read the tables
    keyset_free(ks);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// device-pointer flavour: one launch per call
// ---------------------------------------------------------------------------------------------------
#define DEV_PROLOGUE                                         \
    if (!ctx) return BJJ_ERR_ARG;                            \
    if (n == 0) return BJJ_OK;                               \
    CU(ctx, cudaSetDevice(ctx->device));                     \
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;

// One launch function per operation, shared by the _dev entry point and the host flavour's chunks.  `ws` is the
// scratch of the launch: ctx-wide for _dev calls, per pipeline slot for host calls.
static int launch_fr_op(bjj_ctx* ctx, size_t n, int op, const uint8_t* a, const uint8_t* b, uint8_t* out, cudaStream_t st) {
    k_fr_op<<<grid_for(ctx, k_fr_op, n), BJJ_BLOCK, 0, st>>>(op, n, a, b, out, ctx->flags_dev);
    return launched(ctx);
}
static int launch_split_scalars(bjj_ctx* ctx, size_t n, const uint8_t* h32, const uint8_t* s32, uint8_t* u32, uint8_t* v32,
                                uint8_t* w32, cudaStream_t st) {
    k_split_scalars<<<grid_for(ctx, k_split_scalars, n), BJJ_BLOCK, 0, st>>>(n, h32, s32, u32, v32, w32);
    return launched(ctx);
}
static int launch_add(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz, const uint8_t* qx,
                      const uint8_t* qy, const uint8_t* qz, uint8_t* rx, uint8_t* ry, uint8_t* rz, cudaStream_t st) {
    k_add<<<grid_for(ctx, k_add, n), BJJ_BLOCK, 0, st>>>(n, px, py, pz, qx, qy, qz, rx, ry, rz, ctx->flags_dev);
    return launched(ctx);
}
static int launch_affine(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz, uint8_t* rx,
                         uint8_t* ry, cudaStream_t st) {
    k_affine<<<grid_for(ctx, k_affine, n), BJJ_BLOCK, 0, st>>>(n, px, py, pz, rx, ry, ctx->flags_dev);
    return launched(ctx);
}
static int launch_scalar_key(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* scalar32, cudaStream_t st) {
    k_scalar_key<<<grid_for(ctx, k_scalar_key, n), BJJ_BLOCK, 0, st>>>(n, key32, scalar32);
    return launched(ctx);
}
static int launch_compress(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, uint8_t* out32, cudaStream_t st) {
    k_compress<<<grid_for(ctx, k_compress, n), BJJ_BLOCK, 0, st>>>(n, px, py, out32, ctx->flags_dev);
    return launched(ctx);
}

// k_words = 8: plain 256-bit scalars.  Wider (multiples of 8 words): the on-curve lanes use the scalar reduced mod ORDER
// (k_reduce_scalars), the off-curve lanes replay every bit of the wide scalar.
static int launch_mul_scalar(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* k, int k_words,
                             uint8_t* rx, uint8_t* ry, cudaStream_t st, Workspace* ws) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        const uint8_t* kw = k + (size_t)4 * k_words * off;
        int grid = grid_cap(ctx, bjjk::mul_scalar_blocks_per_sm(), m);
        TRY(ensure_table(ctx, ws, (size_t)grid * BJJ_BLOCK));
        ExactQueue q;
        TRY(ensure_queue(ctx, ws, lanes, st, &q));
        ProjScratch scr;
        TRY(ensure_proj(ctx, ws, lanes, &scr));
        const uint8_t* kfast = kw;
        if (k_words > 8) {
            TRY(grow(ctx, &ws->kred, &ws->kred_lanes, lanes, 32));
            bjjk::reduce_scalars(grid_cap(ctx, 8, m), st, m, kw, k_words, ws->kred);
            TRY(launched(ctx));
            kfast = ws->kred;
        }
        bjjk::mul_scalar(grid, st, m, px + o, py + o, kfast, scr, ws->table, q, ctx->flags_dev);
        TRY(launched(ctx));
        k_batch_affine<<<affine_grid(ctx, m), BJJ_BLOCK, 0, st>>>(m, scr, rx + o, ry + o);
        TRY(launched(ctx));
        bjjk::mul_scalar_exact(ctx->sms * 4, st, px + o, py + o, kw, k_words, rx + o, ry + o, q);
        return launched(ctx);
    });
}
// what the batched affine pass that closes a point sub-batch writes: the (x, y) planes rx, ry (k_batch_affine), or
// Point::compress into the one 32-byte plane rx (k_batch_affine_compressed; ry unused)
enum class PointOut { affine, compressed };

// fixed-base flavours: `from_keys` selects PrivateKey::public (BLAKE-512 + prune + >>3 first)
static int launch_fixed_base(bjj_ctx* ctx, size_t n, const uint8_t* in, uint8_t* rx, uint8_t* ry, bool from_keys,
                             cudaStream_t st, Workspace* ws, PointOut form = PointOut::affine) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        ProjScratch scr;
        TRY(ensure_proj(ctx, ws, lanes, &scr));
        unsigned long long* work = nullptr;
        TRY(claim_counter(ctx, ws, st, &work));
        if (from_keys && ctx->public_fused) {
            k_public<<<grid_for(ctx, k_public, m), BJJ_BLOCK, 0, st>>>(m, in + o, scr, ctx->comb, work);
        } else {
            const uint8_t* k = in + o;
            if (from_keys) {
                // BLAKE-512 is ALU-only work with an 80 KB body: in its own kernel it neither drags the multiplier
                // kernel's instruction supply nor makes ptxas put integer adds on the multiplier pipe.  The scalars pass
                // through the scratch plane that only the batched inversion (afterwards) uses.
                TRY(launch_scalar_key(ctx, m, in + o, scr.p, st));
                k = scr.p;
            }
            k_fixed_base<<<grid_for(ctx, k_fixed_base, m), BJJ_BLOCK, 0, st>>>(m, k, scr, ctx->comb, work);
        }
        TRY(launched(ctx));
        if (form == PointOut::compressed)
            k_batch_affine_compressed<<<affine_grid(ctx, m), BJJ_BLOCK, 0, st>>>(m, scr, rx + o);
        else
            k_batch_affine<<<affine_grid(ctx, m), BJJ_BLOCK, 0, st>>>(m, scr, rx + o, ry + o);
        return launched(ctx);
    });
}
// k * P (l == nullptr) or k * P + l * Q over the tables comb_p, comb_q (bjj_base_mul*)
static int launch_base_mul(bjj_ctx* ctx, size_t n, const uint8_t* k, const uint8_t* l, const CombEntry* comb_p,
                           const CombEntry* comb_q, uint8_t* rx, uint8_t* ry, cudaStream_t st, Workspace* ws) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        ProjScratch scr;
        TRY(ensure_proj(ctx, ws, lanes, &scr));
        unsigned long long* work = nullptr;
        TRY(claim_counter(ctx, ws, st, &work));
        if (l)
            k_fixed_base2<<<grid_for(ctx, k_fixed_base2, m), BJJ_BLOCK, 0, st>>>(m, k + o, l + o, scr, comb_p, comb_q, work);
        else
            k_fixed_base<<<grid_for(ctx, k_fixed_base, m), BJJ_BLOCK, 0, st>>>(m, k + o, scr, comb_p, work);
        TRY(launched(ctx));
        k_batch_affine<<<affine_grid(ctx, m), BJJ_BLOCK, 0, st>>>(m, scr, rx + o, ry + o);
        return launched(ctx);
    });
}
// P_{key_index[i]} * k_i over the compact tables of a key set (bjj_keyset_mul*)
static int launch_keyset_mul(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* key_index, const uint8_t* k, uint8_t* rx,
                             uint8_t* ry, cudaStream_t st, Workspace* ws) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        ProjScratch scr;
        TRY(ensure_proj(ctx, ws, lanes, &scr));
        unsigned long long* work = nullptr;
        TRY(claim_counter(ctx, ws, st, &work));
        k_keyset_mul<<<grid_for(ctx, k_keyset_mul, m), BJJ_BLOCK, 0, st>>>(m, k + o, key_index + 4 * off, (uint32_t)ks->n_keys, ks->tables,
                                                                          scr, ctx->flags_dev, work);
        TRY(launched(ctx));
        k_batch_affine<<<affine_grid(ctx, m), BJJ_BLOCK, 0, st>>>(m, scr, rx + o, ry + o);
        return launched(ctx);
    });
}
// ---- bjj_msm_batch (msm.cuh): begin (clear the buckets), the points in sub-batches, end (reduce, finish) ----------------
// Window width c from n.  c = 16 has 16 + 1 windows against 32 + 1 (half the additions per point) but 2^15 buckets per
// window against 2^7, whose reduction costs the same at any n.  BJJ_MSM_C16_POINTS is the measured crossover (B200,
// 1000 W, profiles/r10_msm.json): c = 8 against c = 16 took 2.26 / 2.30 ms at 2^14 points, 4.74 / 4.80 ms at 2^19,
// 7.60 / 5.86 ms at 2^20 and 13.19 / 10.25 ms at 2^21.  BJJ_MSM_BITS=8 / 16 forces a width (A/B runs of tools/bench_msm.py).
#define BJJ_MSM_C16_POINTS ((size_t)1 << 20)
#define BJJ_MSM_SUBBATCH ((size_t)1 << 20)      // points per prepare / sort / accumulate pass
#define BJJ_MSM_MAX_LEVELS 16
static int msm_window_bits(size_t n) {
    static const int forced = env_int("BJJ_MSM_BITS", 0);
    if (forced == 8 || forced == 16) return forced;
    return n < BJJ_MSM_C16_POINTS ? 8 : 16;
}

// grow() for bjj_msm_batch's scratch: a failed allocation is BJJ_ERR_NOMEM, with the CUDA error cleared
template <class T>
static int msm_grow(bjj_ctx* ctx, T** buf, size_t* cap, size_t want, size_t unit) {
    const int rc = grow(ctx, buf, cap, want, unit);
    if (rc == BJJ_ERR_CUDA && ctx->last == cudaErrorMemoryAllocation) {
        cudaGetLastError();
        ctx->last = cudaSuccess;
        return BJJ_ERR_NOMEM;
    }
    return rc;
}

// the per-call part of the scratch: buckets, segment results, window sums, flags word, result (host flavour)
struct MsmSums {
    uint8_t *buckets, *seg, *wsum, *result;
    uint32_t* flags;
};
static int msm_sums(bjj_ctx* ctx, int bits, MsmSums* out) {
    const MsmGeom g = msm_geom(bits);
    const size_t nb = g.buckets(), segs = (size_t)g.windows * (g.half / BJJ_MSM_SEG);
    TRY(msm_grow(ctx, &ctx->msm.sums, &ctx->msm.sums_cap, 128 * (nb + segs + g.windows) + 128, 1));
    out->buckets = ctx->msm.sums;
    out->seg = out->buckets + 128 * nb;
    out->wsum = out->seg + 128 * segs;
    out->flags = (uint32_t*)(out->wsum + 128 * g.windows);
    out->result = out->wsum + 128 * g.windows + 64;
    return BJJ_OK;
}

// a boundary buffer of `slots` slots: the keys, then (256-byte aligned) the points
static size_t msm_keys_bytes(size_t slots) { return (4 * slots + 255) & ~(size_t)255; }

static int msm_begin(bjj_ctx* ctx, int bits, cudaStream_t st) {
    MsmSums s;
    TRY(msm_sums(ctx, bits, &s));
    CU(ctx, cudaMemsetAsync(s.flags, 0, sizeof(uint32_t), st));
    const size_t nb = msm_geom(bits).buckets();
    bjjk::msm_clear(grid_cap(ctx, 8, nb), st, nb, s.buckets);
    return launched(ctx);
}

// n points into the buckets: per sub-batch prepare, sort, then the accumulate levels (1 + 1 + levels launches; the radix
// sort counts as one)
static int launch_msm_points(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* k, uint8_t* status, int bits,
                             cudaStream_t st) {
    const MsmGeom g = msm_geom(bits);
    const uint32_t nb = g.buckets();
    int key_bits = 1;
    while (((uint32_t)1 << key_bits) <= nb) key_bits++;
    MsmSums s;
    TRY(msm_sums(ctx, bits, &s));
    MsmWork& w = ctx->msm;
    for (size_t off = 0; off < n; off += BJJ_MSM_SUBBATCH) {
        const size_t m = n - off < BJJ_MSM_SUBBATCH ? n - off : BJJ_MSM_SUBBATCH, pairs = m * g.windows;
        size_t counts[BJJ_MSM_MAX_LEVELS];
        const int levels = msm_levels(pairs, counts, BJJ_MSM_MAX_LEVELS);
        const size_t slots0 = 2 * ((pairs + BJJ_MSM_RUN - 1) / BJJ_MSM_RUN), slots1 = levels > 1 ? 2 * ((counts[1] + BJJ_MSM_RUN - 1) / BJJ_MSM_RUN) : 2;
        const size_t temp = bjjk::msm_sort_temp_bytes(pairs, key_bits);
        TRY(msm_grow(ctx, &w.niels, &w.niels_cap, m, sizeof(CombEntry)));
        TRY(msm_grow(ctx, &w.pairs, &w.pairs_cap, 4 * pairs, sizeof(uint32_t)));
        TRY(msm_grow(ctx, &w.sort_temp, &w.sort_temp_cap, temp, 1));
        const size_t slots[2] = {slots0, slots1};
        for (int b = 0; b < 2; b++) TRY(msm_grow(ctx, &w.bound[b], &w.bound_cap[b], msm_keys_bytes(slots[b]) + 128 * slots[b], 1));
        uint8_t* st_out = status ? status + off : nullptr;
        if (!st_out) {
            TRY(msm_grow(ctx, &w.status, &w.status_cap, m, 1));
            st_out = w.status;
        }
        uint32_t* keys[2] = {w.pairs, w.pairs + pairs};
        uint32_t* vals[2] = {w.pairs + 2 * pairs, w.pairs + 3 * pairs};
        bjjk::msm_prepare(grid_cap(ctx, bjjk::msm_prepare_blocks_per_sm(), m), st, m, px + 32 * off, py + 32 * off, k + 32 * off, bits,
                          w.niels, keys[0], vals[0], st_out, s.flags);
        TRY(launched(ctx));
        CU(ctx, bjjk::msm_sort(st, w.sort_temp, temp, keys, vals, pairs, key_bits));
        TRY(launched(ctx));
        // the boundary list that level l writes: bound[l & 1]
        uint32_t* bkeys[2];
        uint8_t* bpts[2];
        for (int b = 0; b < 2; b++) {
            bkeys[b] = (uint32_t*)w.bound[b];
            bpts[b] = w.bound[b] + msm_keys_bytes(slots[b]);
        }
        for (int l = 0; l < levels; l++) {
            const size_t runs = (counts[l] + BJJ_MSM_RUN - 1) / BJJ_MSM_RUN;
            unsigned long long* work = nullptr;
            TRY(claim_counter(ctx, &ctx->ws, st, &work));
            if (l == 0)
                bjjk::msm_accumulate(grid_cap(ctx, bjjk::msm_accumulate_blocks_per_sm(), runs), st, counts[0], keys[0], vals[0], w.niels, nb,
                                     s.buckets, bkeys[0], bpts[0], work);
            else
                bjjk::msm_merge(grid_cap(ctx, bjjk::msm_merge_blocks_per_sm(), runs), st, counts[l], bkeys[(l - 1) & 1], bpts[(l - 1) & 1], nb,
                                s.buckets, bkeys[l & 1], bpts[l & 1], work);
            TRY(launched(ctx));
        }
    }
    return BJJ_OK;
}

// R into (rx, ry), and the call's flags into the context's word (3 launches)
static int msm_end(bjj_ctx* ctx, int bits, uint8_t* rx, uint8_t* ry, cudaStream_t st) {
    const MsmGeom g = msm_geom(bits);
    MsmSums s;
    TRY(msm_sums(ctx, bits, &s));
    const size_t segs = (size_t)g.windows * (g.half / BJJ_MSM_SEG);
    bjjk::msm_bucket_reduce(grid_cap(ctx, bjjk::msm_bucket_reduce_blocks_per_sm(), segs), st, bits, s.buckets, s.seg);
    bjjk::msm_window_sum(st, bits, s.seg, s.wsum);
    bjjk::msm_finish(st, bits, s.wsum, s.flags, rx, ry, ctx->flags_dev);
    return launched(ctx, 3);
}
static int launch_decompress(bjj_ctx* ctx, size_t n, const uint8_t* in32, uint8_t* rx, uint8_t* ry, uint8_t* status,
                             cudaStream_t st, Workspace* ws) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        ProjScratch scr;
        TRY(ensure_proj(ctx, ws, lanes, &scr));
        k_decompress_prepare<<<grid_for(ctx, k_decompress_prepare, m), BJJ_BLOCK, 0, st>>>(m, in32 + o, 1, 0, scr, 0);
        TRY(launched(ctx));
        k_batch_inverse<<<affine_grid(ctx, m), BJJ_BLOCK, 0, st>>>(m, scr);
        TRY(launched(ctx));
        unsigned long long* work = nullptr;
        TRY(claim_counter(ctx, ws, st, &work));
        k_decompress_finish<<<grid_for(ctx, k_decompress_finish, m), BJJ_BLOCK, 0, st>>>(m, in32 + o, 1, 0, scr, 0, rx + o, ry + o,
                                                                                        status + off, 0, work);
        return launched(ctx);
    });
}

// key_index[i] of the key of ks whose compressed bytes are pk32[i], or BJJ_KEY_NONE, for m <= BJJ_POINT_SUBBATCH lanes
static int lookup_subbatch(bjj_ctx* ctx, const bjj_keyset* ks, size_t m, const uint8_t* pk32, uint32_t* key_index, cudaStream_t st,
                           Workspace* ws) {
    unsigned long long* work = nullptr;
    TRY(claim_counter(ctx, ws, st, &work));
    k_keyset_lookup<<<grid_for(ctx, k_keyset_lookup, m), BJJ_BLOCK, 0, st>>>(m, pk32, keyset_comp(ks), keyset_slots(ks), ks->slot_mask,
                                                                            ks->seed, key_index, work);
    return launched(ctx);
}
static int launch_keyset_lookup(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* pk32, uint32_t* key_index, cudaStream_t st,
                                Workspace* ws) {
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        return lookup_subbatch(ctx, ks, m, pk32 + 32 * off, key_index + off, st, ws);
    });
}

// verify scratch: four planes hm | u | v | w (32 B / lane each; u, v, w are the Straus scalars, see split.cuh)
// and, for the compressed pipeline, the four decompressed coordinates
static int ensure_vscratch(bjj_ctx* ctx, Workspace* ws, size_t lanes, uint8_t** hm, uint8_t** pts) {
    TRY(grow(ctx, &ws->vs, &ws->vs_lanes, lanes, 256));
    *hm = ws->vs;
    *pts = ws->vs + 4 * 32 * ws->vs_lanes;
    return BJJ_OK;
}

// mode: BJJ_MODE_EDDSA (verify) or BJJ_MODE_SCHNORR (verify_schnorr; msg_status receives the per-lane Err)
static int launch_verify(bjj_ctx* ctx, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s,
                         const uint8_t* ax, const uint8_t* ay, const uint8_t* msg, uint8_t* ok, cudaStream_t st,
                         Workspace* ws, int mode = BJJ_MODE_EDDSA, uint8_t* msg_status = nullptr, bool defer_join = false) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        const int grid_h = grid_cap(ctx, bjjk::verify_hash_blocks_per_sm(), m);
        const int grid_e = grid_cap(ctx, bjjk::verify_ec_blocks_per_sm(), m);
        TRY(ensure_table(ctx, ws, 2 * (size_t)grid_e * BJJ_BLOCK));     // two per-thread tables: 8A and R8
        TRY(ensure_aux(ctx, ws));
        // exact lanes of an earlier batch may still be reading this workspace's queues and scratch (deferred join):
        // wait for them BEFORE the queue counters are cleared and the scratch is reused
        CU(ctx, cudaStreamWaitEvent(st, ws->ev_join, 0));
        ExactQueue qa, qr;
        TRY(ensure_queue(ctx, ws, lanes, st, &qa, &qr));
        uint8_t *hm, *pts;
        TRY(ensure_vscratch(ctx, ws, lanes, &hm, &pts));
        // BJJ_PHASE_TIMING=1: synchronous per-phase CUDA-event timings on stderr (diagnosis only)
        static const bool phase_timing = getenv("BJJ_PHASE_TIMING") != nullptr;
        cudaEvent_t pe[4] = {nullptr, nullptr, nullptr, nullptr};
        if (phase_timing) {
            for (int e = 0; e < 4; e++) cudaEventCreate(&pe[e]);
            cudaEventRecord(pe[0], st);
        }
        bjjk::verify_hash(grid_h, st, m, r8x + o, r8y + o, ax + o, ay + o, msg + o, s + o, 1, 0, nullptr, hm, ws->vs_lanes, ok + off, true,
                          qa, qr, ctx->flags_dev, mode, ctx->verify_split, msg_status ? msg_status + off : nullptr, work_counters(ws));
        TRY(launched(ctx));
        // The queues are complete after the hash kernel, and the exact lanes (rare; one long ladder each, ~4 % of the
        // step's multiplier work in the benchmark mix) need nothing else: their kernel is released HERE, on the side
        // stream, before the split and the Straus kernel.  Its CTAs are placed first; those that find the queues empty
        // leave at once and the Straus CTAs move into the SMs as they free up (both kernels claim their work
        // dynamically), so the ladders are out of the way early instead of forming a 3-4 ms tail of a few
        // latency-bound warps at the end of the call.  Measured on one GPU (profiles/r2_ab_exact_early_chunks.txt), per
        // 2^21 lanes: 89.5 ms against 90.4 ms with the exact kernel behind the Straus kernel (BJJ_EXACT_EARLY=0, round
        // 1's arrangement).  A small early grid beside the Straus CTAs does not help: the multiplier pipe is the
        // shared limit, Straus + exact take 59.1 ms however they overlap.  All kernels write disjoint ok[] lanes.
        static const int exact_early = env_int("BJJ_EXACT_EARLY", 1);
        static const int exact_ctas = env_int("BJJ_EXACT_CTAS", 8);
        auto launch_exact = [&]() -> int {
            CU(ctx, cudaEventRecord(ws->ev_fork, st));
            CU(ctx, cudaStreamWaitEvent(ws->aux, ws->ev_fork, 0));
            bjjk::verify_exact(ctx->sms * (exact_ctas < 1 ? 1 : exact_ctas), ws->aux, r8x + o, r8y + o, s + o, ax + o, ay + o, hm, ok + off, qa, qr,
                               ctx->comb, mode, work_counters(ws) + 2);
            TRY(launched(ctx));
            CU(ctx, cudaEventRecord(ws->ev_join, ws->aux));
            return BJJ_OK;
        };
        if (exact_early) TRY(launch_exact());
        if (ctx->verify_split && mode == BJJ_MODE_EDDSA) {
            bjjk::verify_split(grid_cap(ctx, bjjk::verify_split_blocks_per_sm(), m), st, m, s + o, 1, 0, hm, ws->vs_lanes, ok + off);
            TRY(launched(ctx));
        }
        if (phase_timing) cudaEventRecord(pe[1], st);
        bjjk::verify_ec(grid_e, st, m, r8x + o, r8y + o, ax + o, ay + o, hm, ws->vs_lanes, ok + off, ws->table, ctx->comb, mode, work_counters(ws) + 1);
        TRY(launched(ctx));
        if (!exact_early) TRY(launch_exact());
        if (phase_timing) cudaEventRecord(pe[2], st);
        // defer_join: the caller orders whatever consumes ok[] after ws->ev_join itself, and the stream moves on
        // to the next batch while the (latency-bound) exact lanes finish beside it
        if (!defer_join) CU(ctx, cudaStreamWaitEvent(st, ws->ev_join, 0));
        if (phase_timing) {
            cudaEventRecord(pe[3], st);
            cudaEventSynchronize(pe[3]);
            float t_hash, t_ec, t_join;
            cudaEventElapsedTime(&t_hash, pe[0], pe[1]);
            cudaEventElapsedTime(&t_ec, pe[1], pe[2]);
            cudaEventElapsedTime(&t_join, pe[2], pe[3]);
            fprintf(stderr, "[bjj phase] lanes=%zu grid_h=%d grid_e=%d hash=%.3f ms ec(+overlapped exact)=%.3f ms join=%.3f ms\n", m, grid_h,
                    grid_e, t_hash, t_ec, t_join);
            for (int e = 0; e < 4; e++) cudaEventDestroy(pe[e]);
        }
        return BJJ_OK;
    });
}
static int launch_verify_compressed(bjj_ctx* ctx, size_t n, const uint8_t* sig64, const uint8_t* pk32,
                                    const uint8_t* msg, uint8_t* ok, uint8_t* status, cudaStream_t st, Workspace* ws) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        const int grid_h = grid_cap(ctx, bjjk::verify_hash_blocks_per_sm(), m);
        const int grid_e = grid_cap(ctx, bjjk::verify_ec_blocks_per_sm(), m);
        TRY(ensure_table(ctx, ws, 2 * (size_t)grid_e * BJJ_BLOCK));
        TRY(ensure_aux(ctx, ws));
        CU(ctx, cudaStreamWaitEvent(st, ws->ev_join, 0));      // a deferred exact kernel of an earlier verify on this workspace
        ExactQueue q;     // never fed here (decompressed points are on the curve) but the kernel wants a valid one
        TRY(ensure_queue(ctx, ws, scratch_lanes(ctx, 1), st, &q));
        uint8_t *hm, *pts;
        TRY(ensure_vscratch(ctx, ws, lanes, &hm, &pts));
        const size_t L = 32 * ws->vs_lanes;
        uint8_t *dx = pts, *dy = pts + L, *dax = pts + 2 * L, *day = pts + 3 * L;
        // phase 0: decompress R8 (first half of each 64-byte signature) and A with one shared inversion pass
        ProjScratch scr;
        TRY(ensure_proj(ctx, ws, 2 * lanes, &scr));       // R8 and A share one inversion pass: two slots per lane
        const int grid_p = grid_for(ctx, k_decompress_prepare, m);
        const int grid_f = grid_for(ctx, k_decompress_finish, m);
        k_decompress_prepare<<<grid_p, BJJ_BLOCK, 0, st>>>(m, sig64 + 2 * o, 2, 0, scr, 0);
        k_decompress_prepare<<<grid_p, BJJ_BLOCK, 0, st>>>(m, pk32 + o, 1, 0, scr, m);
        k_batch_inverse<<<affine_grid(ctx, 2 * m), BJJ_BLOCK, 0, st>>>(2 * m, scr);
        unsigned long long *work_r = nullptr, *work_a = nullptr;
        TRY(claim_counter(ctx, ws, st, &work_r));
        TRY(claim_counter(ctx, ws, st, &work_a));
        k_decompress_finish<<<grid_f, BJJ_BLOCK, 0, st>>>(m, sig64 + 2 * o, 2, 0, scr, 0, dx, dy, status + off, 0, work_r);
        k_decompress_finish<<<grid_f, BJJ_BLOCK, 0, st>>>(m, pk32 + o, 1, 0, scr, m, dax, day, status + off, 1, work_a);
        TRY(launched(ctx, 5));
        bjjk::verify_hash(grid_h, st, m, dx, dy, dax, day, msg + o, sig64 + 2 * o, 2, 1, status + off, hm, ws->vs_lanes, ok + off, false, q,
                          q, ctx->flags_dev, BJJ_MODE_EDDSA, ctx->verify_split, nullptr, work_counters(ws));
        TRY(launched(ctx));
        if (ctx->verify_split) {
            bjjk::verify_split(grid_cap(ctx, bjjk::verify_split_blocks_per_sm(), m), st, m, sig64 + 2 * o, 2, 1, hm, ws->vs_lanes, ok + off);
            TRY(launched(ctx));
        }
        bjjk::verify_ec(grid_e, st, m, dx, dy, dax, day, hm, ws->vs_lanes, ok + off, ws->table, ctx->comb, BJJ_MODE_EDDSA, work_counters(ws) + 1);
        return launched(ctx);
    });
}
// verify against the one key of `base` (bjj_verify_base*): k_verify_base_hash -> k_verify_base_ec, no window tables
// and no exact-lane queue (off-curve R8 lanes take a branch of the EC kernel).  sig64 != nullptr is the compressed
// form: R8 (the first half of each 64-byte signature) is decompressed first into two verify-scratch planes, by phase
// 0 of launch_verify_compressed for R8 alone; `status` receives its decompression status and failed lanes are
// rejected.  The key's coordinates are kernel arguments: base_create checked them.  With a key set `ks` instead of
// `base` (bjj_verify_keyset*), lane i takes key key_index[i] of the set and its compact table: the kernels
// k_verify_keyset_hash -> k_verify_keyset_ec, with the same launches.  s_words != 0 is verify_schnorr
// (bjj_verify_schnorr_base* / _keyset*): r8x, r8y hold r, s32 the signer's s of s_words words per lane, `status` receives
// the msg status, and phase 1 reduces s into the u plane of the verify scratch, which phase 2 reads.  pk32 != nullptr
// (bjj_verify_keyset_lookup_compressed*, with sig64 and ks): after R8's decompression k_keyset_lookup writes the key of
// each lane's compressed key into `found`, which the caller also passes as key_index.  The key-set kernels then raise
// BJJ_FLAG_KEY_INDEX for BJJ_KEY_NONE lanes into the set's own flags word, which nobody reports, instead of the
// context's: an unknown key is data there.  (R8 comes out of decompression canonical, so no other bit can go there.)
static int launch_verify_base(bjj_ctx* ctx, const bjj_base* base, const bjj_keyset* ks, const uint8_t* key_index, size_t n,
                              const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32, const uint8_t* sig64, const uint8_t* msg,
                              uint8_t* ok, uint8_t* status, cudaStream_t st, Workspace* ws, int s_words = 0,
                              const uint8_t* pk32 = nullptr, uint32_t* found = nullptr) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        // the deferred exact kernel of an earlier verify on this workspace may still read its scratch
        if (ws->aux) CU(ctx, cudaStreamWaitEvent(st, ws->ev_join, 0));
        uint8_t *hm, *pts;
        TRY(ensure_vscratch(ctx, ws, lanes, &hm, &pts));
        const uint8_t *rx, *ry, *sb, *skip = nullptr;
        size_t s_stride = 1, s_off = 0;
        if (!sig64) {
            rx = r8x + o;
            ry = r8y + o;
            sb = s32 + o;
        } else {
            uint8_t *dx = pts, *dy = pts + 32 * ws->vs_lanes;
            ProjScratch scr;
            TRY(ensure_proj(ctx, ws, lanes, &scr));
            k_decompress_prepare<<<grid_for(ctx, k_decompress_prepare, m), BJJ_BLOCK, 0, st>>>(m, sig64 + 2 * o, 2, 0, scr, 0);
            k_batch_inverse<<<affine_grid(ctx, m), BJJ_BLOCK, 0, st>>>(m, scr);
            unsigned long long* work = nullptr;
            TRY(claim_counter(ctx, ws, st, &work));
            k_decompress_finish<<<grid_for(ctx, k_decompress_finish, m), BJJ_BLOCK, 0, st>>>(m, sig64 + 2 * o, 2, 0, scr, 0, dx, dy,
                                                                                            status + off, 0, work);
            TRY(launched(ctx, 3));
            rx = dx;
            ry = dy;
            sb = sig64 + 2 * o;
            s_stride = 2;
            s_off = 1;
            skip = status + off;
        }
        if (pk32) TRY(lookup_subbatch(ctx, ks, m, pk32 + o, found + off, st, ws));
        unsigned long long *work_h = nullptr, *work_e = nullptr;
        TRY(claim_counter(ctx, ws, st, &work_h));
        TRY(claim_counter(ctx, ws, st, &work_e));
        if (s_words) {
            uint8_t* sred = hm + 32 * ws->vs_lanes;
            const SchnorrWide sw{s32 + (size_t)4 * s_words * off, s_words, sred, status + off};
            if (ks) {
                const uint8_t *ki = key_index + 4 * off, *kx = ks->keys, *ky = kx + 32 * ks->n_keys;
                const uint32_t nk = (uint32_t)ks->n_keys;
                bjjk::verify_schnorr_keyset_hash(grid_cap(ctx, bjjk::verify_schnorr_keyset_hash_blocks_per_sm(), m), st, m, rx, ry, ki, kx, ky,
                                                 nk, msg + o, sw, hm, ok + off, ctx->flags_dev, work_h);
                TRY(launched(ctx));
                bjjk::verify_schnorr_keyset_ec(grid_cap(ctx, bjjk::verify_schnorr_keyset_ec_blocks_per_sm(), m), st, m, rx, ry, sred, hm,
                                               ok + off, ctx->comb, ki, nk, ks->tables, work_e);
                return launched(ctx);
            }
            bjjk::verify_schnorr_base_hash(grid_cap(ctx, bjjk::verify_schnorr_base_hash_blocks_per_sm(), m), st, m, rx, ry, base->x, base->y,
                                           msg + o, sw, hm, ok + off, ctx->flags_dev, work_h);
            TRY(launched(ctx));
            bjjk::verify_schnorr_base_ec(grid_cap(ctx, bjjk::verify_schnorr_base_ec_blocks_per_sm(), m), st, m, rx, ry, sred, hm, ok + off,
                                         ctx->comb, base->comb, work_e);
            return launched(ctx);
        }
        if (ks) {
            const uint8_t *ki = key_index + 4 * off, *kx = ks->keys, *ky = kx + 32 * ks->n_keys;
            const uint32_t nk = (uint32_t)ks->n_keys;
            bjjk::verify_keyset_hash(grid_cap(ctx, bjjk::verify_keyset_hash_blocks_per_sm(), m), st, m, rx, ry, ki, kx, ky, nk, msg + o,
                                     skip, hm, ok + off, pk32 ? keyset_quiet_flags(ks) : ctx->flags_dev, work_h);
            TRY(launched(ctx));
            bjjk::verify_keyset_ec(grid_cap(ctx, bjjk::verify_keyset_ec_blocks_per_sm(), m), st, m, rx, ry, sb, s_stride, s_off, hm,
                                   ok + off, ctx->comb, ki, nk, ks->tables, work_e);
            return launched(ctx);
        }
        bjjk::verify_base_hash(grid_cap(ctx, bjjk::verify_base_hash_blocks_per_sm(), m), st, m, rx, ry, base->x, base->y, msg + o, skip,
                               hm, ok + off, ctx->flags_dev, work_h);
        TRY(launched(ctx));
        bjjk::verify_base_ec(grid_cap(ctx, bjjk::verify_base_ec_blocks_per_sm(), m), st, m, rx, ry, sb, s_stride, s_off, hm, ok + off,
                             ctx->comb, base->comb, work_e);
        return launched(ctx);
    });
}
// verify_schnorr with s at the signer's width on the Straus path (bjj_verify_schnorr_wide*): per sub-batch,
// k_mod_suborder_wide reduces s into the first decompressed-point plane of the verify scratch (launch_verify's plain
// form does not use it), then launch_verify runs unchanged with that plane as s.
static int launch_verify_schnorr_wide(bjj_ctx* ctx, size_t n, const uint8_t* pkx, const uint8_t* pky, const uint8_t* msg,
                                      const uint8_t* rx, const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok, uint8_t* status,
                                      cudaStream_t st, Workspace* ws, bool defer_join = false) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        // the deferred exact kernel of an earlier verify on this workspace may still read the plane
        if (ws->aux) CU(ctx, cudaStreamWaitEvent(st, ws->ev_join, 0));
        uint8_t *hm, *sred;
        TRY(ensure_vscratch(ctx, ws, lanes, &hm, &sred));
        k_mod_suborder_wide<<<grid_for(ctx, k_mod_suborder_wide, m), BJJ_BLOCK, 0, st>>>(m, s + (size_t)4 * s_words * off, s_words, sred);
        TRY(launched(ctx));
        return launch_verify(ctx, m, rx + o, ry + o, sred, pkx + o, pky + o, msg + o, ok + off, st, ws, BJJ_MODE_SCHNORR, status + off,
                             defer_join);
    });
}
// the widths of s that bjj_verify_schnorr_{base,keyset,wide}* take: those bjj_sign_schnorr_batch writes (nonce_words + 8)
static bool s_words_ok(int w) { return w >= 8 && w <= BJJ_MAX_SCALAR_WORDS + 8 && !(w & 7); }

// a verify_base call names its key: NULL or a handle of another context is an argument error
static bool base_of(bjj_ctx* ctx, const bjj_base* base) { return base && base->ctx == ctx; }

static int launch_poseidon(bjj_ctx* ctx, int n_inputs, size_t n, const uint8_t* const* in, uint8_t* out,
                           cudaStream_t st) {
    PoseidonIn pin;
    for (int j = 0; j < 8; j++) pin.p[j] = j < n_inputs ? in[j] : nullptr;
    if (n_inputs < 1 || n_inputs > BJJ_POSEIDON_MAX_INPUTS) return BJJ_ERR_ARG;
    bjjk::poseidon(n_inputs + 1, grid_cap(ctx, bjjk::poseidon_blocks_per_sm(n_inputs + 1), n), st, n, pin, out, ctx->flags_dev);
    return launched(ctx);
}

// PrivateKey::sign as a pipeline: k_sign_scalars (BLAKE-512 twice: sk, r) -> R8 = r * B8 and A = sk * B8 on the
// fixed-base kernels with batched inversions -> hm = Poseidon(R8, A, msg) on k_poseidon<6> -> k_sign_finish (S).  The
// fused k_sign (one lane start to finish in one thread: 244 registers with spills, a Fermat inversion per lane, 67 % of
// the multiplier pipe) stays available as BJJ_SIGN_FUSED=1; the pipeline reuses kernels that run at 84-92 %.
// form == PointOut::compressed writes Signature::compress into the 64-byte-stride array r8x (r8y and s32 unused) and
// always runs the pipeline: R8's affine coordinates then go to the two verify-scratch planes that signing leaves free,
// and k_sign_finish_compressed packs compress(R8) || S.
static int launch_sign(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* r8x, uint8_t* r8y, uint8_t* s32,
                       uint8_t* status, cudaStream_t st, Workspace* ws, PointOut form = PointOut::affine) {
    const bool packed = form == PointOut::compressed;
    if (ctx->sign_fused && !packed) {
        bjjk::sign(grid_cap(ctx, bjjk::sign_blocks_per_sm(), n), st, n, key32, msg32, r8x, r8y, s32, status, ctx->comb);
        return launched(ctx);
    }
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        uint8_t *hm, *pts;
        TRY(ensure_vscratch(ctx, ws, lanes, &hm, &pts));
        const size_t L = 32 * ws->vs_lanes;
        uint8_t *sk = hm + L, *r = hm + 2 * L, *msgc = hm + 3 * L, *apx = pts, *apy = pts + L;
        uint8_t *rx = packed ? pts + 2 * L : r8x + o, *ry = packed ? pts + 3 * L : r8y + o;
        const int grid_s = grid_for(ctx, k_scalar_key, m);      // same block size and shape of work
        bjjk::sign_scalars(grid_s, st, m, key32 + o, msg32 + o, sk, r, msgc, status + off);
        TRY(launched(ctx));
        TRY(launch_fixed_base(ctx, m, r, rx, ry, false, st, ws));
        TRY(launch_fixed_base(ctx, m, sk, apx, apy, false, st, ws));
        const uint8_t* ins[5] = {rx, ry, apx, apy, msgc};
        TRY(launch_poseidon(ctx, 5, m, ins, hm, st));
        if (packed)
            bjjk::sign_finish_compressed(grid_s, st, m, hm, sk, r, status + off, rx, ry, r8x + 2 * o);
        else
            bjjk::sign_finish(grid_s, st, m, hm, sk, r, status + off, rx, ry, s32 + o);
        return launched(ctx);
    });
}

// PrivateKey::sign_schnorr with caller nonces, shaped like launch_sign: k_sign_schnorr_scalars (BLAKE-512 once: sk; the
// nonce mod SUBORDER: kr) -> r = kr * B8 straight into the caller's planes and pk = sk * B8 on the fixed-base kernels ->
// h = Poseidon(pk, r, msg) on k_poseidon<6> -> k_sign_schnorr_finish (s = k + sk * h, exact).  sk, kr, msgc, h, pk.x and
// pk.y take six of the eight verify-scratch planes.  The nonce and s advance by their own strides (4 * nonce_words and
// 4 * (nonce_words + 8) bytes per lane).
static int launch_sign_schnorr(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, const uint8_t* nonce,
                               int nonce_words, uint8_t* rx, uint8_t* ry, uint8_t* s, uint8_t* status, cudaStream_t st,
                               Workspace* ws) {
    const size_t lanes = scratch_lanes(ctx, n);
    return for_each_subbatch(n, [&](size_t off, size_t m) -> int {
        const size_t o = 32 * off;
        const uint8_t* k = nonce + (size_t)4 * nonce_words * off;
        uint8_t* so = s + (size_t)4 * (nonce_words + 8) * off;
        // the deferred exact kernel of an earlier verify on this workspace may still read its scratch
        if (ws->aux) CU(ctx, cudaStreamWaitEvent(st, ws->ev_join, 0));
        uint8_t *h, *pts;
        TRY(ensure_vscratch(ctx, ws, lanes, &h, &pts));
        const size_t L = 32 * ws->vs_lanes;
        uint8_t *sk = h + L, *kr = h + 2 * L, *msgc = h + 3 * L, *pkx = pts, *pky = pts + L;
        const int grid_s = grid_for(ctx, k_scalar_key, m);      // same block size and shape of work
        bjjk::sign_schnorr_scalars(grid_s, st, m, key32 + o, msg32 + o, k, nonce_words, sk, kr, msgc, status + off);
        TRY(launched(ctx));
        TRY(launch_fixed_base(ctx, m, kr, rx + o, ry + o, false, st, ws));
        TRY(launch_fixed_base(ctx, m, sk, pkx, pky, false, st, ws));
        const uint8_t* ins[5] = {pkx, pky, rx + o, ry + o, msgc};
        TRY(launch_poseidon(ctx, 5, m, ins, h, st));
        bjjk::sign_schnorr_finish(grid_s, st, m, h, sk, k, nonce_words, status + off, rx + o, ry + o, so);
        return launched(ctx);
    });
}
// the nonce widths of bjj_sign_schnorr_batch: those of bjj_mul_scalar_wide_batch
static bool nonce_words_ok(int w) { return w >= 8 && w <= BJJ_MAX_SCALAR_WORDS && !(w & 7); }

extern "C" {

int bjj_fr_op_batch_dev(bjj_ctx* ctx, int op, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out, void* stream) {
    DEV_PROLOGUE
    if (!a || !out || op < 0 || op > BJJ_FR_SQR_LAZY) return BJJ_ERR_ARG;
    if (!b) b = a;
    return launch_fr_op(ctx, n, op, a, b, out, st);
}

int bjj_split_scalars_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* h32, const uint8_t* s32, uint8_t* u32,
                                uint8_t* v32, uint8_t* w32, void* stream) {
    DEV_PROLOGUE
    if (!h32 || !s32 || !u32 || !v32 || !w32) return BJJ_ERR_ARG;
    return launch_split_scalars(ctx, n, h32, s32, u32, v32, w32, st);
}

int bjj_add_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz,
                      const uint8_t* qx, const uint8_t* qy, const uint8_t* qz, uint8_t* rx, uint8_t* ry, uint8_t* rz,
                      void* stream) {
    DEV_PROLOGUE
    if (!px || !py || !pz || !qx || !qy || !qz || !rx || !ry || !rz) return BJJ_ERR_ARG;
    return launch_add(ctx, n, px, py, pz, qx, qy, qz, rx, ry, rz, st);
}

int bjj_affine_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz, uint8_t* rx,
                         uint8_t* ry, void* stream) {
    DEV_PROLOGUE
    if (!px || !py || !pz || !rx || !ry) return BJJ_ERR_ARG;
    return launch_affine(ctx, n, px, py, pz, rx, ry, st);
}

int bjj_mul_scalar_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32,
                             uint8_t* rx, uint8_t* ry, void* stream) {
    DEV_PROLOGUE
    if (!px || !py || !scalar32 || !rx || !ry) return BJJ_ERR_ARG;
    return launch_mul_scalar(ctx, n, px, py, scalar32, 8, rx, ry, st, &ctx->ws);
}

int bjj_mul_scalar_wide_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar, int scalar_words,
                                  uint8_t* rx, uint8_t* ry, void* stream) {
    DEV_PROLOGUE
    if (!px || !py || !scalar || !rx || !ry || scalar_words < 8 || scalar_words > BJJ_MAX_SCALAR_WORDS || (scalar_words & 7)) return BJJ_ERR_ARG;
    return launch_mul_scalar(ctx, n, px, py, scalar, scalar_words, rx, ry, st, &ctx->ws);
}

int bjj_fixed_base_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry, void* stream) {
    DEV_PROLOGUE
    if (!scalar32 || !rx || !ry) return BJJ_ERR_ARG;
    return launch_fixed_base(ctx, n, scalar32, rx, ry, false, st, &ctx->ws);
}

int bjj_public_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* rx, uint8_t* ry, void* stream) {
    DEV_PROLOGUE
    if (!key32 || !rx || !ry) return BJJ_ERR_ARG;
    return launch_fixed_base(ctx, n, key32, rx, ry, true, st, &ctx->ws);
}

int bjj_public_compressed_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* out32, void* stream) {
    DEV_PROLOGUE
    if (!key32 || !out32) return BJJ_ERR_ARG;
    return launch_fixed_base(ctx, n, key32, out32, nullptr, true, st, &ctx->ws, PointOut::compressed);
}

int bjj_base_mul_batch_dev(bjj_ctx* ctx, const bjj_base* base, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry,
                           void* stream) {
    DEV_PROLOGUE
    const CombEntry* comb = base_comb(ctx, base);
    if (!comb || !scalar32 || !rx || !ry) return BJJ_ERR_ARG;
    return launch_base_mul(ctx, n, scalar32, nullptr, comb, nullptr, rx, ry, st, &ctx->ws);
}

int bjj_base_mul2_batch_dev(bjj_ctx* ctx, const bjj_base* p, const bjj_base* q, size_t n, const uint8_t* k32,
                            const uint8_t* l32, uint8_t* rx, uint8_t* ry, void* stream) {
    DEV_PROLOGUE
    const CombEntry *comb_p = base_comb(ctx, p), *comb_q = base_comb(ctx, q);
    if (!comb_p || !comb_q || !k32 || !l32 || !rx || !ry) return BJJ_ERR_ARG;
    return launch_base_mul(ctx, n, k32, l32, comb_p, comb_q, rx, ry, st, &ctx->ws);
}

int bjj_sign_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* r8x, uint8_t* r8y,
                       uint8_t* s32, uint8_t* status, void* stream) {
    DEV_PROLOGUE
    if (!key32 || !msg32 || !r8x || !r8y || !s32 || !status) return BJJ_ERR_ARG;
    return launch_sign(ctx, n, key32, msg32, r8x, r8y, s32, status, st, &ctx->ws);
}

int bjj_sign_compressed_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* sig64,
                                  uint8_t* status, void* stream) {
    DEV_PROLOGUE
    if (!key32 || !msg32 || !sig64 || !status) return BJJ_ERR_ARG;
    return launch_sign(ctx, n, key32, msg32, sig64, nullptr, nullptr, status, st, &ctx->ws, PointOut::compressed);
}

int bjj_sign_schnorr_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, const uint8_t* nonce,
                               int nonce_words, uint8_t* rx, uint8_t* ry, uint8_t* s, uint8_t* status, void* stream) {
    DEV_PROLOGUE
    if (!key32 || !msg32 || !nonce || !nonce_words_ok(nonce_words) || !rx || !ry || !s || !status) return BJJ_ERR_ARG;
    return launch_sign_schnorr(ctx, n, key32, msg32, nonce, nonce_words, rx, ry, s, status, st, &ctx->ws);
}

int bjj_scalar_key_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* scalar32, void* stream) {
    DEV_PROLOGUE
    if (!key32 || !scalar32) return BJJ_ERR_ARG;
    return launch_scalar_key(ctx, n, key32, scalar32, st);
}

int bjj_compress_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, uint8_t* out32, void* stream) {
    DEV_PROLOGUE
    if (!px || !py || !out32) return BJJ_ERR_ARG;
    return launch_compress(ctx, n, px, py, out32, st);
}

int bjj_decompress_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* in32, uint8_t* rx, uint8_t* ry, uint8_t* status,
                             void* stream) {
    DEV_PROLOGUE
    if (!in32 || !rx || !ry || !status) return BJJ_ERR_ARG;
    return launch_decompress(ctx, n, in32, rx, ry, status, st, &ctx->ws);
}

int bjj_poseidon_batch_dev(bjj_ctx* ctx, int n_inputs, size_t n, const uint8_t* const* in, uint8_t* out, void* stream) {
    DEV_PROLOGUE
    if (!in || !out || n_inputs < 1 || n_inputs > BJJ_POSEIDON_MAX_INPUTS) return BJJ_ERR_ARG;
    for (int j = 0; j < n_inputs; j++)
        if (!in[j]) return BJJ_ERR_ARG;
    return launch_poseidon(ctx, n_inputs, n, in, out, st);
}

int bjj_verify_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32,
                         const uint8_t* ax, const uint8_t* ay, const uint8_t* msg32, uint8_t* ok, void* stream) {
    DEV_PROLOGUE
    if (!r8x || !r8y || !s32 || !ax || !ay || !msg32 || !ok) return BJJ_ERR_ARG;
    return launch_verify(ctx, n, r8x, r8y, s32, ax, ay, msg32, ok, st, &ctx->ws);
}

int bjj_verify_schnorr_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* pkx, const uint8_t* pky, const uint8_t* msg32,
                                 const uint8_t* rx, const uint8_t* ry, const uint8_t* s32, uint8_t* ok, uint8_t* status,
                                 void* stream) {
    DEV_PROLOGUE
    if (!pkx || !pky || !msg32 || !rx || !ry || !s32 || !ok || !status) return BJJ_ERR_ARG;
    return launch_verify(ctx, n, rx, ry, s32, pkx, pky, msg32, ok, st, &ctx->ws, BJJ_MODE_SCHNORR, status);
}

int bjj_verify_compressed_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* sig64, const uint8_t* pk32,
                                    const uint8_t* msg32, uint8_t* ok, uint8_t* status, void* stream) {
    DEV_PROLOGUE
    if (!sig64 || !pk32 || !msg32 || !ok || !status) return BJJ_ERR_ARG;
    return launch_verify_compressed(ctx, n, sig64, pk32, msg32, ok, status, st, &ctx->ws);
}

int bjj_verify_base_batch_dev(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* r8x, const uint8_t* r8y,
                              const uint8_t* s32, const uint8_t* msg32, uint8_t* ok, void* stream) {
    if (!base_of(ctx, pk)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!r8x || !r8y || !s32 || !msg32 || !ok) return BJJ_ERR_ARG;
    return launch_verify_base(ctx, pk, nullptr, nullptr, n, r8x, r8y, s32, nullptr, msg32, ok, nullptr, st, &ctx->ws);
}

int bjj_verify_base_compressed_batch_dev(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* sig64, const uint8_t* msg32,
                                         uint8_t* ok, uint8_t* status, void* stream) {
    if (!base_of(ctx, pk)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!sig64 || !msg32 || !ok || !status) return BJJ_ERR_ARG;
    return launch_verify_base(ctx, pk, nullptr, nullptr, n, nullptr, nullptr, nullptr, sig64, msg32, ok, status, st, &ctx->ws);
}

int bjj_verify_keyset_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* r8x,
                                const uint8_t* r8y, const uint8_t* s32, const uint8_t* msg32, uint8_t* ok, void* stream) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!key_index || !r8x || !r8y || !s32 || !msg32 || !ok) return BJJ_ERR_ARG;
    return launch_verify_base(ctx, nullptr, ks, (const uint8_t*)key_index, n, r8x, r8y, s32, nullptr, msg32, ok, nullptr, st, &ctx->ws);
}

int bjj_verify_keyset_compressed_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index,
                                           const uint8_t* sig64, const uint8_t* msg32, uint8_t* ok, uint8_t* status, void* stream) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!key_index || !sig64 || !msg32 || !ok || !status) return BJJ_ERR_ARG;
    return launch_verify_base(ctx, nullptr, ks, (const uint8_t*)key_index, n, nullptr, nullptr, nullptr, sig64, msg32, ok, status, st,
                              &ctx->ws);
}

int bjj_keyset_mul_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* scalar32,
                             uint8_t* rx, uint8_t* ry, void* stream) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!key_index || !scalar32 || !rx || !ry) return BJJ_ERR_ARG;
    return launch_keyset_mul(ctx, ks, n, (const uint8_t*)key_index, scalar32, rx, ry, st, &ctx->ws);
}

int bjj_keyset_lookup_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* pk32, uint32_t* key_index, void* stream) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!pk32 || !key_index) return BJJ_ERR_ARG;
    return launch_keyset_lookup(ctx, ks, n, pk32, key_index, st, &ctx->ws);
}

int bjj_verify_keyset_lookup_compressed_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* sig64, const uint8_t* pk32,
                                                  const uint8_t* msg32, uint8_t* ok, uint8_t* status, uint32_t* key_index, void* stream) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!sig64 || !pk32 || !msg32 || !ok || !status || !key_index) return BJJ_ERR_ARG;
    return launch_verify_base(ctx, nullptr, ks, (const uint8_t*)key_index, n, nullptr, nullptr, nullptr, sig64, msg32, ok, status, st,
                              &ctx->ws, 0, pk32, key_index);
}

int bjj_msm_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32, uint8_t* rx32, uint8_t* ry32,
                      uint8_t* point_status, void* stream) {
    if (!ctx || !px || !py || !scalar32 || !rx32 || !ry32) return BJJ_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = stream ? (cudaStream_t)stream : ctx->stream;
    const int bits = msm_window_bits(n);
    TRY(msm_begin(ctx, bits, st));
    TRY(launch_msm_points(ctx, n, px, py, scalar32, point_status, bits, st));
    return msm_end(ctx, bits, rx32, ry32, st);
}

int bjj_verify_schnorr_base_batch_dev(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* msg32, const uint8_t* rx,
                                      const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok, uint8_t* status, void* stream) {
    if (!base_of(ctx, pk) || !s_words_ok(s_words)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!msg32 || !rx || !ry || !s || !ok || !status) return BJJ_ERR_ARG;
    return launch_verify_base(ctx, pk, nullptr, nullptr, n, rx, ry, s, nullptr, msg32, ok, status, st, &ctx->ws, s_words);
}

int bjj_verify_schnorr_keyset_batch_dev(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* msg32,
                                        const uint8_t* rx, const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok, uint8_t* status,
                                        void* stream) {
    if (!keyset_of(ctx, ks) || !s_words_ok(s_words)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!key_index || !msg32 || !rx || !ry || !s || !ok || !status) return BJJ_ERR_ARG;
    return launch_verify_base(ctx, nullptr, ks, (const uint8_t*)key_index, n, rx, ry, s, nullptr, msg32, ok, status, st, &ctx->ws,
                              s_words);
}

int bjj_verify_schnorr_wide_batch_dev(bjj_ctx* ctx, size_t n, const uint8_t* pkx, const uint8_t* pky, const uint8_t* msg32,
                                      const uint8_t* rx, const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok, uint8_t* status,
                                      void* stream) {
    if (!s_words_ok(s_words)) return BJJ_ERR_ARG;
    DEV_PROLOGUE
    if (!pkx || !pky || !msg32 || !rx || !ry || !s || !ok || !status) return BJJ_ERR_ARG;
    return launch_verify_schnorr_wide(ctx, n, pkx, pky, msg32, rx, ry, s, s_words, ok, status, st, &ctx->ws);
}

}  // extern "C"

// ---------------------------------------------------------------------------------------------------
// host-pointer flavour: chunked, double-buffered H2D -> kernel -> D2H pipeline over two streams
// ---------------------------------------------------------------------------------------------------
struct HostArg {
    const uint8_t* in;    // non-null for inputs
    uint8_t* out;         // non-null for outputs
    size_t bytes_per_lane;
};

// Copies and kernels overlap, kernels never overlap each other: every kernel of this library is sized to fill
// the GPU and streams a large instruction footprint, and two of them sharing SMs starve each other's
// instruction fetch (measured: two concurrent verify pipelines ran at 0.65x the serial rate; round 2, odd chunks on a
// second compute stream so that the block scheduler could fill one chunk's kernel tails with the next chunk's
// kernels: 17.8 against 22.7 M verifies/s end to end, profiles/r2_ab_exact_early_chunks.txt).  So the two slots
// only own copy streams and staging arenas; all launches go to the context's one compute stream, ordered against
// the copies by events.  Chunk sizes ramp up from 2^18 lanes so that only the first, small host-to-device copy is
// exposed (shape: see below).
template <class Launch>
static int run_host(bjj_ctx* ctx, size_t n, HostArg* args, int nargs, Launch launch, bool heavy = false) {
    if (!ctx) return BJJ_ERR_ARG;
    for (int a = 0; a < nargs; a++)
        if (!args[a].in && !args[a].out) return BJJ_ERR_ARG;
    if (n == 0) return BJJ_OK;
    CU(ctx, cudaSetDevice(ctx->device));
    // Which caller arrays are pageable?  (cudaHostAlloc'd / cudaHostRegister'ed ones go to the copy engine directly.)
    static const int stage_pageable = env_int("BJJ_STAGE_PAGEABLE", 1);
    bool staged[16];
    bool any_staged = false;
    for (int a = 0; a < nargs; a++) {
        cudaPointerAttributes at;
        const void* hp = args[a].in ? (const void*)args[a].in : (const void*)args[a].out;
        const cudaError_t e = cudaPointerGetAttributes(&at, hp);
        if (e != cudaSuccess) cudaGetLastError();
        staged[a] = stage_pageable && (e != cudaSuccess || at.type == cudaMemoryTypeUnregistered);
        any_staged = any_staged || staged[a];
    }
    for (int k = 0; k < BJJ_PIPE_SLOTS; k++) ctx->slot[k].drain_pending = false;      // (an aborted call may have left one)
    // Chunk shape.  Every chunk boundary costs the tails of its kernels (the last wave of the Straus kernel alone is
    // ~2.5 ms), so the compute-heavy calls (`heavy`: verify*, mul_scalar* -- tens of ns of arithmetic per lane against
    // ~4 ns of PCIe) go from the small first chunk straight to chunks of 2^21 lanes: the copy of a chunk eight times
    // larger still ends before the kernels of the one before it.  The copy-bound calls keep the gentle ramp and the
    // smaller chunk, whose last copy-out is the exposed part.  BJJ_CHUNK_LOG2 / BJJ_CHUNK_GROWTH override (A/B runs).
    static const int env_log2 = env_int("BJJ_CHUNK_LOG2", 0), env_growth = env_int("BJJ_CHUNK_GROWTH", 0);
    const size_t chunk_max = env_log2 >= 16 && env_log2 <= 24 ? (size_t)1 << env_log2 : (heavy ? BJJ_POINT_SUBBATCH : (size_t)BJJ_CHUNK_LANES);
    // (staged, i.e. pageable, arrays: the calling thread's memcpy of the next chunk, ~20 ns per verify lane, has to fit
    // under the kernels of this one, ~43 ns per lane -- so those calls double instead)
    const size_t growth = env_growth >= 2 ? (size_t)env_growth : (heavy && !any_staged ? 8 : 2);
    const size_t chunk = n < chunk_max ? n : chunk_max;
    // a chunk may grow by half when the lanes left over after it would make a short, inefficient last chunk -- but not
    // past the sub-batch of the point kernels, which would split it into two sets of launches again
    size_t cap = chunk + chunk / 2;
    if (cap > BJJ_POINT_SUBBATCH && chunk <= BJJ_POINT_SUBBATCH) cap = BJJ_POINT_SUBBATCH;
    // every array slice starts 256-byte aligned inside the arena
    size_t need = 0;
    for (int a = 0; a < nargs; a++) need += ((args[a].bytes_per_lane * cap + 255) & ~(size_t)255);
    int rc = BJJ_OK;
    int which = 0;
    // verify_compressed parks two points per lane in the projective scratch: the hint covers the larger user
    ctx->lane_hint = cap <= 2 * BJJ_POINT_SUBBATCH ? cap : 0;
    struct HintReset {
        bjj_ctx* c;
        ~HintReset() { c->lane_hint = 0; }
    } hint_reset{ctx};
    // BJJ_PIPE_TIMING=1: per-chunk timeline (ms since the call started) on stderr -- diagnosis only
    static const bool pipe_timing = getenv("BJJ_PIPE_TIMING") != nullptr;
    struct Mark { cudaEvent_t in, comp, out; size_t lanes; };
    Mark marks[64];
    int nmarks = 0;
    cudaEvent_t t0 = nullptr;
    if (pipe_timing) {
        cudaEventCreate(&t0);
        cudaEventRecord(t0, ctx->stream);
    }
    // copies a drained slot's outputs from its page-locked mirror to the caller's (pageable) arrays
    auto drain = [&](PipeSlot& sl) -> int {
        if (!sl.drain_pending) return BJJ_OK;
        CU(ctx, cudaEventSynchronize(sl.ev_done));
        size_t pos = 0;
        for (int a = 0; a < nargs; a++) {
            if (args[a].out && staged[a])
                memcpy(args[a].out + sl.drain_off * args[a].bytes_per_lane, sl.hstage + pos, sl.drain_lanes * args[a].bytes_per_lane);
            pos += ((args[a].bytes_per_lane * cap + 255) & ~(size_t)255);
        }
        sl.drain_pending = false;
        return BJJ_OK;
    };
    size_t cur = n > 2 * BJJ_CHUNK_RAMP_LANES && chunk > BJJ_CHUNK_RAMP_LANES ? BJJ_CHUNK_RAMP_LANES : chunk;
    size_t m = 0;
    for (size_t off = 0; off < n; off += m, which ^= 1, cur = (growth * cur < chunk ? growth * cur : chunk)) {
        PipeSlot& sl = ctx->slot[which];
        m = (n - off) < cur ? (n - off) : cur;
        if (n - off - m < cur / 2 && n - off <= cap) m = n - off;      // fold a short remainder into this chunk
        // the slot's copies of two chunks ago may still use the arena and the mirror: let them finish before a regrowth
        if (sl.arena_bytes < need) CU(ctx, cudaStreamSynchronize(sl.stream));
        TRY(grow(ctx, &sl.arena, &sl.arena_bytes, need, 1));
        if (any_staged) {
            // the slot's previous chunk: its results go out to the caller, and its host-to-device copies have long
            // finished reading the mirror (they precede ev_done on the slot's stream)
            rc = drain(sl);
            if (rc) break;
            if (sl.hstage_bytes < need) CU(ctx, cudaStreamSynchronize(sl.stream));
            TRY(grow(ctx, &sl.hstage, &sl.hstage_bytes, need, 1, /*pinned=*/true));
        }
        // the slot's copy stream is ordered: these copies follow the slot's previous results going out
        uint8_t* dptr[16];
        size_t pos = 0;
        for (int a = 0; a < nargs; a++) {
            dptr[a] = sl.arena + pos;
            if (args[a].in) {
                const uint8_t* src = args[a].in + off * args[a].bytes_per_lane;
                if (staged[a]) {
                    memcpy(sl.hstage + pos, src, m * args[a].bytes_per_lane);
                    src = sl.hstage + pos;
                }
                CU(ctx, cudaMemcpyAsync(dptr[a], src, m * args[a].bytes_per_lane, cudaMemcpyHostToDevice, sl.stream));
            }
            pos += ((args[a].bytes_per_lane * cap + 255) & ~(size_t)255);
        }
        Workspace* ws = which ? &ctx->ws2 : &ctx->ws;
        CU(ctx, cudaEventRecord(sl.ev_in, sl.stream));
        const bool mark = pipe_timing && nmarks < 64;
        if (mark) {
            Mark& mk = marks[nmarks];
            cudaEventCreate(&mk.in);
            cudaEventCreate(&mk.comp);
            cudaEventCreate(&mk.out);
            mk.lanes = m;
            cudaEventRecord(mk.in, sl.stream);
        }
        CU(ctx, cudaStreamWaitEvent(ctx->stream, sl.ev_in, 0));
        rc = launch(m, dptr, ctx->stream, ws);
        if (rc) break;
        if (mark) cudaEventRecord(marks[nmarks].comp, ctx->stream);
        CU(ctx, cudaEventRecord(sl.ev_out, ctx->stream));
        CU(ctx, cudaStreamWaitEvent(sl.stream, sl.ev_out, 0));
        if (ws->aux) CU(ctx, cudaStreamWaitEvent(sl.stream, ws->ev_join, 0));      // deferred exact lanes
        pos = 0;
        for (int a = 0; a < nargs; a++) {
            if (args[a].out)
                CU(ctx, cudaMemcpyAsync(staged[a] ? sl.hstage + pos : args[a].out + off * args[a].bytes_per_lane, dptr[a],
                                        m * args[a].bytes_per_lane, cudaMemcpyDeviceToHost, sl.stream));
            pos += ((args[a].bytes_per_lane * cap + 255) & ~(size_t)255);
        }
        if (any_staged) {
            CU(ctx, cudaEventRecord(sl.ev_done, sl.stream));
            sl.drain_pending = true;
            sl.drain_off = off;
            sl.drain_lanes = m;
        }
        if (mark) cudaEventRecord(marks[nmarks++].out, sl.stream);
    }
    if (rc) {
        // copies and kernels of earlier chunks may still be in flight against the caller's buffers: drain them before
        // handing the buffers back
        bjj_sync(ctx);
        for (int k = 0; k < BJJ_PIPE_SLOTS; k++) ctx->slot[k].drain_pending = false;
        return rc;
    }
    for (int k = 0; k < BJJ_PIPE_SLOTS; k++) {       // oldest first: `which` now names the slot used two chunks ago
        const int r2 = drain(ctx->slot[which ^ k]);
        if (r2 && !rc) rc = r2;
    }
    if (rc) {
        bjj_sync(ctx);
        return rc;
    }
    rc = bjj_sync(ctx);
    if (pipe_timing) {
        for (int k = 0; k < nmarks; k++) {
            float a = 0, b = 0, d = 0;
            cudaEventElapsedTime(&a, t0, marks[k].in);
            cudaEventElapsedTime(&b, t0, marks[k].comp);
            cudaEventElapsedTime(&d, t0, marks[k].out);
            fprintf(stderr, "[bjj pipe] chunk %d lanes=%zu copied-in at %.2f ms, kernels done at %.2f ms, copied-out at %.2f ms\n", k,
                    marks[k].lanes, a, b, d);
            cudaEventDestroy(marks[k].in);
            cudaEventDestroy(marks[k].comp);
            cudaEventDestroy(marks[k].out);
        }
        cudaEventDestroy(t0);
    }
    return rc;
}

#define H_IN(p, b) HostArg{(p), nullptr, (b)}
#define H_OUT(p, b) HostArg{nullptr, (p), (b)}

extern "C" {

int bjj_fr_op_batch(bjj_ctx* ctx, int op, size_t n, const uint8_t* a, const uint8_t* b, uint8_t* out) {
    if (!ctx || !a || !out || op < 0 || op > BJJ_FR_SQR_LAZY) return BJJ_ERR_ARG;
    if (!b) b = a;
    HostArg args[] = {H_IN(a, 32), H_IN(b, 32), H_OUT(out, 32)};
    return run_host(ctx, n, args, 3, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_fr_op(ctx, m, op, d[0], d[1], d[2], st);
    });
}

int bjj_split_scalars_batch(bjj_ctx* ctx, size_t n, const uint8_t* h32, const uint8_t* s32, uint8_t* u32, uint8_t* v32,
                            uint8_t* w32) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(h32, 32), H_IN(s32, 32), H_OUT(u32, 32), H_OUT(v32, 32), H_OUT(w32, 32)};
    return run_host(ctx, n, args, 5, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_split_scalars(ctx, m, d[0], d[1], d[2], d[3], d[4], st);
    });
}

int bjj_add_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz, const uint8_t* qx,
                  const uint8_t* qy, const uint8_t* qz, uint8_t* rx, uint8_t* ry, uint8_t* rz) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(px, 32), H_IN(py, 32), H_IN(pz, 32), H_IN(qx, 32), H_IN(qy, 32),
                      H_IN(qz, 32), H_OUT(rx, 32), H_OUT(ry, 32), H_OUT(rz, 32)};
    return run_host(ctx, n, args, 9, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_add(ctx, m, d[0], d[1], d[2], d[3], d[4], d[5], d[6], d[7], d[8], st);
    });
}

int bjj_affine_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* pz, uint8_t* rx,
                     uint8_t* ry) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(px, 32), H_IN(py, 32), H_IN(pz, 32), H_OUT(rx, 32), H_OUT(ry, 32)};
    return run_host(ctx, n, args, 5, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_affine(ctx, m, d[0], d[1], d[2], d[3], d[4], st);
    });
}

int bjj_mul_scalar_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32,
                         uint8_t* rx, uint8_t* ry) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(px, 32), H_IN(py, 32), H_IN(scalar32, 32), H_OUT(rx, 32), H_OUT(ry, 32)};
    return run_host(ctx, n, args, 5, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_mul_scalar(ctx, m, d[0], d[1], d[2], 8, d[3], d[4], st, ws);
    }, /*heavy=*/true);
}

int bjj_mul_scalar_wide_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar, int scalar_words,
                              uint8_t* rx, uint8_t* ry) {
    if (!ctx || scalar_words < 8 || scalar_words > BJJ_MAX_SCALAR_WORDS || (scalar_words & 7)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(px, 32), H_IN(py, 32), H_IN(scalar, (size_t)4 * scalar_words), H_OUT(rx, 32), H_OUT(ry, 32)};
    return run_host(ctx, n, args, 5, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_mul_scalar(ctx, m, d[0], d[1], d[2], scalar_words, d[3], d[4], st, ws);
    }, /*heavy=*/true);
}

int bjj_fixed_base_batch(bjj_ctx* ctx, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(scalar32, 32), H_OUT(rx, 32), H_OUT(ry, 32)};
    return run_host(ctx, n, args, 3, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_fixed_base(ctx, m, d[0], d[1], d[2], false, st, ws);
    });
}

int bjj_public_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* rx, uint8_t* ry) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(key32, 32), H_OUT(rx, 32), H_OUT(ry, 32)};
    return run_host(ctx, n, args, 3, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_fixed_base(ctx, m, d[0], d[1], d[2], true, st, ws);
    });
}

int bjj_public_compressed_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* out32) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(key32, 32), H_OUT(out32, 32)};
    return run_host(ctx, n, args, 2, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_fixed_base(ctx, m, d[0], d[1], nullptr, true, st, ws, PointOut::compressed);
    });
}

int bjj_base_mul_batch(bjj_ctx* ctx, const bjj_base* base, size_t n, const uint8_t* scalar32, uint8_t* rx, uint8_t* ry) {
    if (!ctx) return BJJ_ERR_ARG;
    const CombEntry* comb = base_comb(ctx, base);
    if (!comb) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(scalar32, 32), H_OUT(rx, 32), H_OUT(ry, 32)};
    return run_host(ctx, n, args, 3, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_base_mul(ctx, m, d[0], nullptr, comb, nullptr, d[1], d[2], st, ws);
    });
}

int bjj_base_mul2_batch(bjj_ctx* ctx, const bjj_base* p, const bjj_base* q, size_t n, const uint8_t* k32, const uint8_t* l32,
                        uint8_t* rx, uint8_t* ry) {
    if (!ctx) return BJJ_ERR_ARG;
    const CombEntry *comb_p = base_comb(ctx, p), *comb_q = base_comb(ctx, q);
    if (!comb_p || !comb_q) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(k32, 32), H_IN(l32, 32), H_OUT(rx, 32), H_OUT(ry, 32)};
    return run_host(ctx, n, args, 4, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_base_mul(ctx, m, d[0], d[1], comb_p, comb_q, d[2], d[3], st, ws);
    });
}

int bjj_sign_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* r8x, uint8_t* r8y,
                   uint8_t* s32, uint8_t* status) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(key32, 32), H_IN(msg32, 32), H_OUT(r8x, 32), H_OUT(r8y, 32), H_OUT(s32, 32), H_OUT(status, 1)};
    return run_host(ctx, n, args, 6, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_sign(ctx, m, d[0], d[1], d[2], d[3], d[4], d[5], st, ws);
    });
}

int bjj_sign_compressed_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, uint8_t* sig64,
                              uint8_t* status) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(key32, 32), H_IN(msg32, 32), H_OUT(sig64, 64), H_OUT(status, 1)};
    return run_host(ctx, n, args, 4, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_sign(ctx, m, d[0], d[1], d[2], nullptr, nullptr, d[3], st, ws, PointOut::compressed);
    });
}

int bjj_sign_schnorr_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, const uint8_t* msg32, const uint8_t* nonce, int nonce_words,
                           uint8_t* rx, uint8_t* ry, uint8_t* s, uint8_t* status) {
    if (!ctx || !nonce_words_ok(nonce_words)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(key32, 32), H_IN(msg32, 32), H_IN(nonce, (size_t)4 * nonce_words), H_OUT(rx, 32), H_OUT(ry, 32),
                      H_OUT(s, (size_t)4 * (nonce_words + 8)), H_OUT(status, 1)};
    return run_host(ctx, n, args, 7, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_sign_schnorr(ctx, m, d[0], d[1], d[2], nonce_words, d[3], d[4], d[5], d[6], st, ws);
    });
}

int bjj_scalar_key_batch(bjj_ctx* ctx, size_t n, const uint8_t* key32, uint8_t* scalar32) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(key32, 32), H_OUT(scalar32, 32)};
    return run_host(ctx, n, args, 2, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_scalar_key(ctx, m, d[0], d[1], st);
    });
}

int bjj_compress_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, uint8_t* out32) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(px, 32), H_IN(py, 32), H_OUT(out32, 32)};
    return run_host(ctx, n, args, 3, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_compress(ctx, m, d[0], d[1], d[2], st);
    });
}

int bjj_decompress_batch(bjj_ctx* ctx, size_t n, const uint8_t* in32, uint8_t* rx, uint8_t* ry, uint8_t* status) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(in32, 32), H_OUT(rx, 32), H_OUT(ry, 32), H_OUT(status, 1)};
    return run_host(ctx, n, args, 4, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_decompress(ctx, m, d[0], d[1], d[2], d[3], st, ws);
    });
}

int bjj_poseidon_batch(bjj_ctx* ctx, int n_inputs, size_t n, const uint8_t* const* in, uint8_t* out) {
    if (!ctx || !in || n_inputs < 1 || n_inputs > BJJ_POSEIDON_MAX_INPUTS) return BJJ_ERR_ARG;
    HostArg args[9];
    for (int j = 0; j < n_inputs; j++) args[j] = H_IN(in[j], 32);
    args[n_inputs] = H_OUT(out, 32);
    return run_host(ctx, n, args, n_inputs + 1, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_poseidon(ctx, n_inputs, m, (const uint8_t* const*)d, d[n_inputs], st);
    });
}

int bjj_verify_batch(bjj_ctx* ctx, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32,
                     const uint8_t* ax, const uint8_t* ay, const uint8_t* msg32, uint8_t* ok) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(r8x, 32), H_IN(r8y, 32), H_IN(s32, 32), H_IN(ax, 32), H_IN(ay, 32), H_IN(msg32, 32), H_OUT(ok, 1)};
    return run_host(ctx, n, args, 7, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify(ctx, m, d[0], d[1], d[2], d[3], d[4], d[5], d[6], st, ws, BJJ_MODE_EDDSA, nullptr, true);
    }, /*heavy=*/true);
}

int bjj_verify_schnorr_batch(bjj_ctx* ctx, size_t n, const uint8_t* pkx, const uint8_t* pky, const uint8_t* msg32,
                             const uint8_t* rx, const uint8_t* ry, const uint8_t* s32, uint8_t* ok, uint8_t* status) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(pkx, 32), H_IN(pky, 32), H_IN(msg32, 32), H_IN(rx, 32), H_IN(ry, 32), H_IN(s32, 32), H_OUT(ok, 1),
                      H_OUT(status, 1)};
    return run_host(ctx, n, args, 8, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify(ctx, m, d[3], d[4], d[5], d[0], d[1], d[2], d[6], st, ws, BJJ_MODE_SCHNORR, d[7], true);
    }, /*heavy=*/true);
}

int bjj_verify_compressed_batch(bjj_ctx* ctx, size_t n, const uint8_t* sig64, const uint8_t* pk32,
                                const uint8_t* msg32, uint8_t* ok, uint8_t* status) {
    if (!ctx) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(sig64, 64), H_IN(pk32, 32), H_IN(msg32, 32), H_OUT(ok, 1), H_OUT(status, 1)};
    return run_host(ctx, n, args, 5, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify_compressed(ctx, m, d[0], d[1], d[2], d[3], d[4], st, ws);
    }, /*heavy=*/true);
}

int bjj_verify_base_batch(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32,
                          const uint8_t* msg32, uint8_t* ok) {
    if (!base_of(ctx, pk)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(r8x, 32), H_IN(r8y, 32), H_IN(s32, 32), H_IN(msg32, 32), H_OUT(ok, 1)};
    return run_host(ctx, n, args, 5, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify_base(ctx, pk, nullptr, nullptr, m, d[0], d[1], d[2], nullptr, d[3], d[4], nullptr, st, ws);
    }, /*heavy=*/true);
}

int bjj_verify_base_compressed_batch(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* sig64, const uint8_t* msg32,
                                     uint8_t* ok, uint8_t* status) {
    if (!base_of(ctx, pk)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(sig64, 64), H_IN(msg32, 32), H_OUT(ok, 1), H_OUT(status, 1)};
    return run_host(ctx, n, args, 4, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify_base(ctx, pk, nullptr, nullptr, m, nullptr, nullptr, nullptr, d[0], d[1], d[2], d[3], st, ws);
    }, /*heavy=*/true);
}

int bjj_verify_keyset_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* r8x,
                            const uint8_t* r8y, const uint8_t* s32, const uint8_t* msg32, uint8_t* ok) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN((const uint8_t*)key_index, 4), H_IN(r8x, 32), H_IN(r8y, 32), H_IN(s32, 32), H_IN(msg32, 32), H_OUT(ok, 1)};
    return run_host(ctx, n, args, 6, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify_base(ctx, nullptr, ks, d[0], m, d[1], d[2], d[3], nullptr, d[4], d[5], nullptr, st, ws);
    }, /*heavy=*/true);
}

int bjj_verify_keyset_compressed_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* sig64,
                                       const uint8_t* msg32, uint8_t* ok, uint8_t* status) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN((const uint8_t*)key_index, 4), H_IN(sig64, 64), H_IN(msg32, 32), H_OUT(ok, 1), H_OUT(status, 1)};
    return run_host(ctx, n, args, 5, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify_base(ctx, nullptr, ks, d[0], m, nullptr, nullptr, nullptr, d[1], d[2], d[3], d[4], st, ws);
    }, /*heavy=*/true);
}

int bjj_keyset_mul_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* scalar32, uint8_t* rx,
                         uint8_t* ry) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN((const uint8_t*)key_index, 4), H_IN(scalar32, 32), H_OUT(rx, 32), H_OUT(ry, 32)};
    return run_host(ctx, n, args, 4, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_keyset_mul(ctx, ks, m, d[0], d[1], d[2], d[3], st, ws);
    }, /*heavy=*/true);
}

int bjj_keyset_lookup_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* pk32, uint32_t* key_index) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(pk32, 32), H_OUT((uint8_t*)key_index, 4)};
    return run_host(ctx, n, args, 2, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_keyset_lookup(ctx, ks, m, d[0], (uint32_t*)d[1], st, ws);
    });
}

int bjj_verify_keyset_lookup_compressed_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint8_t* sig64, const uint8_t* pk32,
                                              const uint8_t* msg32, uint8_t* ok, uint8_t* status, uint32_t* key_index) {
    if (!keyset_of(ctx, ks)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(sig64, 64), H_IN(pk32, 32), H_IN(msg32, 32), H_OUT(ok, 1), H_OUT(status, 1), H_OUT((uint8_t*)key_index, 4)};
    return run_host(ctx, n, args, 6, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify_base(ctx, nullptr, ks, d[5], m, nullptr, nullptr, nullptr, d[0], d[2], d[3], d[4], st, ws, 0, d[1],
                                  (uint32_t*)d[5]);
    }, /*heavy=*/true);
}

int bjj_msm_batch(bjj_ctx* ctx, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* scalar32, uint8_t* rx32, uint8_t* ry32,
                  uint8_t* point_status) {
    if (!ctx || !px || !py || !scalar32 || !rx32 || !ry32) return BJJ_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    std::vector<uint8_t> own_status;
    if (!point_status) {
        own_status.resize(n ? n : 1);
        point_status = own_status.data();
    }
    const int bits = msm_window_bits(n);
    TRY(msm_begin(ctx, bits, ctx->stream));
    // every chunk adds into the same buckets; the reduction and the one inversion follow the last chunk
    HostArg args[] = {H_IN(px, 32), H_IN(py, 32), H_IN(scalar32, 32), H_OUT(point_status, 1)};
    TRY(run_host(ctx, n, args, 4, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace*) -> int {
        return launch_msm_points(ctx, m, d[0], d[1], d[2], d[3], bits, st);
    }, /*heavy=*/true));
    MsmSums s;
    TRY(msm_sums(ctx, bits, &s));
    TRY(msm_end(ctx, bits, s.result, s.result + 32, ctx->stream));
    CU(ctx, cudaMemcpyAsync(rx32, s.result, 32, cudaMemcpyDeviceToHost, ctx->stream));
    CU(ctx, cudaMemcpyAsync(ry32, s.result + 32, 32, cudaMemcpyDeviceToHost, ctx->stream));
    return bjj_sync(ctx);
}

int bjj_verify_schnorr_base_batch(bjj_ctx* ctx, const bjj_base* pk, size_t n, const uint8_t* msg32, const uint8_t* rx, const uint8_t* ry,
                                  const uint8_t* s, int s_words, uint8_t* ok, uint8_t* status) {
    if (!base_of(ctx, pk) || !s_words_ok(s_words)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(msg32, 32), H_IN(rx, 32), H_IN(ry, 32), H_IN(s, (size_t)4 * s_words), H_OUT(ok, 1), H_OUT(status, 1)};
    return run_host(ctx, n, args, 6, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify_base(ctx, pk, nullptr, nullptr, m, d[1], d[2], d[3], nullptr, d[0], d[4], d[5], st, ws, s_words);
    }, /*heavy=*/true);
}

int bjj_verify_schnorr_keyset_batch(bjj_ctx* ctx, const bjj_keyset* ks, size_t n, const uint32_t* key_index, const uint8_t* msg32,
                                    const uint8_t* rx, const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok, uint8_t* status) {
    if (!keyset_of(ctx, ks) || !s_words_ok(s_words)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN((const uint8_t*)key_index, 4), H_IN(msg32, 32), H_IN(rx, 32),    H_IN(ry, 32),
                      H_IN(s, (size_t)4 * s_words),       H_OUT(ok, 1),      H_OUT(status, 1)};
    return run_host(ctx, n, args, 7, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify_base(ctx, nullptr, ks, d[0], m, d[2], d[3], d[4], nullptr, d[1], d[5], d[6], st, ws, s_words);
    }, /*heavy=*/true);
}

int bjj_verify_schnorr_wide_batch(bjj_ctx* ctx, size_t n, const uint8_t* pkx, const uint8_t* pky, const uint8_t* msg32, const uint8_t* rx,
                                  const uint8_t* ry, const uint8_t* s, int s_words, uint8_t* ok, uint8_t* status) {
    if (!ctx || !s_words_ok(s_words)) return BJJ_ERR_ARG;
    HostArg args[] = {H_IN(pkx, 32), H_IN(pky, 32), H_IN(msg32, 32), H_IN(rx, 32), H_IN(ry, 32), H_IN(s, (size_t)4 * s_words), H_OUT(ok, 1),
                      H_OUT(status, 1)};
    return run_host(ctx, n, args, 8, [&](size_t m, uint8_t** d, cudaStream_t st, Workspace* ws) -> int {
        return launch_verify_schnorr_wide(ctx, m, d[0], d[1], d[2], d[3], d[4], d[5], s_words, d[6], d[7], st, ws, true);
    }, /*heavy=*/true);
}

}  // extern "C"
