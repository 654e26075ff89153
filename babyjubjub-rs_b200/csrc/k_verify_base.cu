// verify_base_batch / verify_base_compressed_batch kernels: verify (src/lib.rs:395-412) for a batch signed by ONE key A
// with a comb table (bjj_base_create).  The lane bodies and their exactness argument are in lanes.cuh
// (lane_verify_base_hash, lane_verify_base_ec).
//
//   (bjj_cuda.cu: k_decompress_prepare / k_batch_inverse / k_decompress_finish for compressed R8) ->
//   k_verify_base_hash -> k_verify_base_ec       (one key, bjj_verify_base*)
//   k_verify_keyset_hash -> k_verify_keyset_ec   (a key per lane from a key set, bjj_verify_keyset*)
//   k_verify_schnorr_base_hash -> k_verify_schnorr_base_ec       (verify_schnorr, one key, bjj_verify_schnorr_base*)
//   k_verify_schnorr_keyset_hash -> k_verify_schnorr_keyset_ec   (verify_schnorr, key set, bjj_verify_schnorr_keyset*)
#include "kernels.h"

using namespace bjj;

// A's canonical affine coordinates as a kernel argument (the same for every lane)
struct BaseKey {
    uint32_t x[8], y[8];
};

__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_verify_base_hash(size_t n, const uint8_t* r8x, const uint8_t* r8y, BaseKey key,
                                                                   const uint8_t* msg, const uint8_t* skip, uint8_t* hm, uint8_t* ok,
                                                                   uint32_t* gflags, unsigned long long* work) {
    BJJ_FLAGS_BEGIN
    PointAff a;
    {
        Fr raw;
        fr_set(raw, key.x);
        fr_to_mont(a.x, raw);
        fr_set(raw, key.y);
        fr_to_mont(a.y, raw);
    }
    BJJ_CLAIM_LOOP(n, work)
    if (i < n) lane_verify_base_hash(r8x, r8y, a, msg, skip, hm, ok, i, flags);
    BJJ_FLAGS_END(gflags)
}

__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_verify_base_ec(size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s_base,
                                                                 size_t s_stride, size_t s_off, const uint8_t* hm, uint8_t* ok,
                                                                 const CombEntry* comb, const CombEntry* comb_a,
                                                                 unsigned long long* work) {
    BJJ_CLAIM_LOOP(n, work)
    if (i < n) lane_verify_base_ec(r8x, r8y, s_base, s_stride, s_off, hm, ok, i, comb, comb_a);
}

// the same two phases against a key set: key key_index[i] of the set serves lane i (lanes.cuh: lane_verify_keyset_*)
__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_verify_keyset_hash(size_t n, const uint8_t* r8x, const uint8_t* r8y,
                                                                     const uint8_t* key_index, const uint8_t* kx, const uint8_t* ky,
                                                                     uint32_t n_keys, const uint8_t* msg, const uint8_t* skip,
                                                                     uint8_t* hm, uint8_t* ok, uint32_t* gflags,
                                                                     unsigned long long* work) {
    BJJ_FLAGS_BEGIN
    BJJ_CLAIM_LOOP(n, work)
    if (i < n) lane_verify_keyset_hash(r8x, r8y, key_index, kx, ky, n_keys, msg, skip, hm, ok, i, flags);
    BJJ_FLAGS_END(gflags)
}

__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_verify_keyset_ec(size_t n, const uint8_t* r8x, const uint8_t* r8y,
                                                                   const uint8_t* s_base, size_t s_stride, size_t s_off,
                                                                   const uint8_t* hm, uint8_t* ok, const CombEntry* comb,
                                                                   const uint8_t* key_index, uint32_t n_keys,
                                                                   const CombEntry* tables, unsigned long long* work) {
    BJJ_CLAIM_LOOP(n, work)
    if (i < n) lane_verify_keyset_ec(r8x, r8y, s_base, s_stride, s_off, hm, ok, i, comb, key_index, n_keys, tables);
}

// verify_schnorr on the same phases (lanes.cuh: SchnorrWide): phase 1 also reduces the signer's wide s into sw.s_out and
// writes every lane's msg status; phase 2 reads that reduced s (32 B per lane)
__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_verify_schnorr_base_hash(size_t n, const uint8_t* rx, const uint8_t* ry, BaseKey key,
                                                                           const uint8_t* msg, SchnorrWide sw, uint8_t* hm, uint8_t* ok,
                                                                           uint32_t* gflags, unsigned long long* work) {
    BJJ_FLAGS_BEGIN
    PointAff a;
    {
        Fr raw;
        fr_set(raw, key.x);
        fr_to_mont(a.x, raw);
        fr_set(raw, key.y);
        fr_to_mont(a.y, raw);
    }
    BJJ_CLAIM_LOOP(n, work)
    if (i < n) lane_verify_base_hash<BJJ_MODE_SCHNORR>(rx, ry, a, msg, nullptr, hm, ok, i, flags, sw);
    BJJ_FLAGS_END(gflags)
}

__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_verify_schnorr_base_ec(size_t n, const uint8_t* rx, const uint8_t* ry,
                                                                         const uint8_t* s_red, const uint8_t* hm, uint8_t* ok,
                                                                         const CombEntry* comb, const CombEntry* comb_a,
                                                                         unsigned long long* work) {
    BJJ_CLAIM_LOOP(n, work)
    if (i < n) lane_verify_base_ec<Comb16, BJJ_MODE_SCHNORR>(rx, ry, s_red, 1, 0, hm, ok, i, comb, comb_a);
}

__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_verify_schnorr_keyset_hash(size_t n, const uint8_t* rx, const uint8_t* ry,
                                                                             const uint8_t* key_index, const uint8_t* kx,
                                                                             const uint8_t* ky, uint32_t n_keys, const uint8_t* msg,
                                                                             SchnorrWide sw, uint8_t* hm, uint8_t* ok, uint32_t* gflags,
                                                                             unsigned long long* work) {
    BJJ_FLAGS_BEGIN
    BJJ_CLAIM_LOOP(n, work)
    if (i < n) lane_verify_keyset_hash<BJJ_MODE_SCHNORR>(rx, ry, key_index, kx, ky, n_keys, msg, nullptr, hm, ok, i, flags, sw);
    BJJ_FLAGS_END(gflags)
}

__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_verify_schnorr_keyset_ec(size_t n, const uint8_t* rx, const uint8_t* ry,
                                                                           const uint8_t* s_red, const uint8_t* hm, uint8_t* ok,
                                                                           const CombEntry* comb, const uint8_t* key_index,
                                                                           uint32_t n_keys, const CombEntry* tables,
                                                                           unsigned long long* work) {
    BJJ_CLAIM_LOOP(n, work)
    if (i < n) lane_verify_keyset_ec<BJJ_MODE_SCHNORR>(rx, ry, s_red, 1, 0, hm, ok, i, comb, key_index, n_keys, tables);
}

namespace bjjk {

void verify_base_hash(int grid, cudaStream_t st, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* ax32,
                      const uint8_t* ay32, const uint8_t* msg, const uint8_t* skip, uint8_t* hm, uint8_t* ok, uint32_t* gflags,
                      unsigned long long* work) {
    BaseKey key;
    memcpy(key.x, ax32, 32);
    memcpy(key.y, ay32, 32);
    k_verify_base_hash<<<grid, BJJ_BLOCK, 0, st>>>(n, r8x, r8y, key, msg, skip, hm, ok, gflags, work);
}
int verify_base_hash_blocks_per_sm() { return blocks_per_sm(k_verify_base_hash); }

void verify_base_ec(int grid, cudaStream_t st, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s_base,
                    size_t s_stride, size_t s_off, const uint8_t* hm, uint8_t* ok, const bjj::CombEntry* comb,
                    const bjj::CombEntry* comb_a, unsigned long long* work) {
    k_verify_base_ec<<<grid, BJJ_BLOCK, 0, st>>>(n, r8x, r8y, s_base, s_stride, s_off, hm, ok, comb, comb_a, work);
}
int verify_base_ec_blocks_per_sm() { return blocks_per_sm(k_verify_base_ec); }

void verify_keyset_hash(int grid, cudaStream_t st, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* key_index,
                        const uint8_t* kx, const uint8_t* ky, uint32_t n_keys, const uint8_t* msg, const uint8_t* skip, uint8_t* hm,
                        uint8_t* ok, uint32_t* gflags, unsigned long long* work) {
    k_verify_keyset_hash<<<grid, BJJ_BLOCK, 0, st>>>(n, r8x, r8y, key_index, kx, ky, n_keys, msg, skip, hm, ok, gflags, work);
}
int verify_keyset_hash_blocks_per_sm() { return blocks_per_sm(k_verify_keyset_hash); }

void verify_keyset_ec(int grid, cudaStream_t st, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s_base,
                      size_t s_stride, size_t s_off, const uint8_t* hm, uint8_t* ok, const bjj::CombEntry* comb,
                      const uint8_t* key_index, uint32_t n_keys, const bjj::CombEntry* tables, unsigned long long* work) {
    k_verify_keyset_ec<<<grid, BJJ_BLOCK, 0, st>>>(n, r8x, r8y, s_base, s_stride, s_off, hm, ok, comb, key_index, n_keys, tables, work);
}
int verify_keyset_ec_blocks_per_sm() { return blocks_per_sm(k_verify_keyset_ec); }

void verify_schnorr_base_hash(int grid, cudaStream_t st, size_t n, const uint8_t* rx, const uint8_t* ry, const uint8_t* pkx32,
                              const uint8_t* pky32, const uint8_t* msg, const bjj::SchnorrWide& sw, uint8_t* hm, uint8_t* ok,
                              uint32_t* gflags, unsigned long long* work) {
    BaseKey key;
    memcpy(key.x, pkx32, 32);
    memcpy(key.y, pky32, 32);
    k_verify_schnorr_base_hash<<<grid, BJJ_BLOCK, 0, st>>>(n, rx, ry, key, msg, sw, hm, ok, gflags, work);
}
int verify_schnorr_base_hash_blocks_per_sm() { return blocks_per_sm(k_verify_schnorr_base_hash); }

void verify_schnorr_base_ec(int grid, cudaStream_t st, size_t n, const uint8_t* rx, const uint8_t* ry, const uint8_t* s_red,
                            const uint8_t* hm, uint8_t* ok, const bjj::CombEntry* comb, const bjj::CombEntry* comb_a,
                            unsigned long long* work) {
    k_verify_schnorr_base_ec<<<grid, BJJ_BLOCK, 0, st>>>(n, rx, ry, s_red, hm, ok, comb, comb_a, work);
}
int verify_schnorr_base_ec_blocks_per_sm() { return blocks_per_sm(k_verify_schnorr_base_ec); }

void verify_schnorr_keyset_hash(int grid, cudaStream_t st, size_t n, const uint8_t* rx, const uint8_t* ry, const uint8_t* key_index,
                                const uint8_t* kx, const uint8_t* ky, uint32_t n_keys, const uint8_t* msg, const bjj::SchnorrWide& sw,
                                uint8_t* hm, uint8_t* ok, uint32_t* gflags, unsigned long long* work) {
    k_verify_schnorr_keyset_hash<<<grid, BJJ_BLOCK, 0, st>>>(n, rx, ry, key_index, kx, ky, n_keys, msg, sw, hm, ok, gflags, work);
}
int verify_schnorr_keyset_hash_blocks_per_sm() { return blocks_per_sm(k_verify_schnorr_keyset_hash); }

void verify_schnorr_keyset_ec(int grid, cudaStream_t st, size_t n, const uint8_t* rx, const uint8_t* ry, const uint8_t* s_red,
                              const uint8_t* hm, uint8_t* ok, const bjj::CombEntry* comb, const uint8_t* key_index, uint32_t n_keys,
                              const bjj::CombEntry* tables, unsigned long long* work) {
    k_verify_schnorr_keyset_ec<<<grid, BJJ_BLOCK, 0, st>>>(n, rx, ry, s_red, hm, ok, comb, key_index, n_keys, tables, work);
}
int verify_schnorr_keyset_ec_blocks_per_sm() { return blocks_per_sm(k_verify_schnorr_keyset_ec); }

}  // namespace bjjk
