// Host-callable launch wrappers of the heavy kernels.  Each heavy kernel lives in its own translation
// unit (k_*.cu) so that the library builds in parallel; bjj_cuda.cu holds the light kernels, the
// context and the C ABI.  A wrapper does exactly one <<<...>>> launch on the given stream.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "lanes.cuh"

#define BJJ_BLOCK 128
#define BJJ_EXACT_BLOCK 64

#define BJJ_LANE_LOOP(n) \
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < (n); i += (size_t)gridDim.x * blockDim.x)
// Dynamic lane assignment: a warp claims 32 consecutive lanes at a time from a device counter (zeroed before the
// launch).  A CTA that becomes resident late -- the exact-lane kernel of the previous batch may still hold
// registers on its SM -- then simply takes less work, where a grid-stride split would make the whole kernel
// wait for it.
#if defined(__CUDACC__)
__device__ __forceinline__ size_t bjj_claim_lanes(unsigned long long* counter) {
    unsigned long long b = 0;
    if ((threadIdx.x & 31) == 0) b = atomicAdd(counter, 32ull);
    return (size_t)__shfl_sync(0xFFFFFFFFu, b, 0) + (threadIdx.x & 31);
}
#endif
#define BJJ_CLAIM_LOOP(n, counter) for (size_t i = bjj_claim_lanes(counter); i - (threadIdx.x & 31) < (n); i = bjj_claim_lanes(counter))
#define BJJ_QUEUE_LOOP(q) \
    for (uint32_t j = blockIdx.x * blockDim.x + threadIdx.x, cnt = *(q).count; j < cnt; j += gridDim.x * blockDim.x)
#define BJJ_FLAGS_BEGIN uint32_t flags = 0;
#define BJJ_FLAGS_END(p) \
    if (flags) atomicOr(p, flags);

#if defined(__CUDACC__)
__device__ __forceinline__ bjj::LaneTable thread_table(bjj::U128* base) {
    bjj::LaneTable t;
    t.base = base;
    t.stride = (size_t)gridDim.x * blockDim.x;
    t.slot = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    return t;
}
#endif

struct PoseidonIn {
    const uint8_t* p[8];
};

namespace bjjk {

// resident CTAs per SM of `kernel` launched with `block` threads and `smem` bytes of dynamic shared memory, >= 1
template <class Kernel>
inline int blocks_per_sm(Kernel* kernel, int block = BJJ_BLOCK, size_t smem = 0) {
    int per_sm = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void*)kernel, block, smem) != cudaSuccess || per_sm < 1)
        per_sm = 1;
    return per_sm;
}

// blocks_per_sm of the kernels behind the launch wrappers below
int verify_hash_blocks_per_sm();
int verify_ec_blocks_per_sm();
int verify_split_blocks_per_sm();
int mul_scalar_blocks_per_sm();
int sign_blocks_per_sm();
int poseidon_blocks_per_sm(int t);

void verify_hash(int grid, cudaStream_t st, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* ax,
                 const uint8_t* ay, const uint8_t* msg, const uint8_t* s_base, size_t s_stride, size_t s_off,
                 const uint8_t* skip, uint8_t* hm, size_t plane, uint8_t* ok, bool gate, bjj::ExactQueue qa,
                 bjj::ExactQueue qr, uint32_t* gflags, int mode, bool split, uint8_t* msg_status, unsigned long long* work);
void verify_split(int grid, cudaStream_t st, size_t n, const uint8_t* s_base, size_t s_stride, size_t s_off, uint8_t* hm,
                  size_t plane, const uint8_t* ok);
void verify_ec(int grid, cudaStream_t st, size_t n, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* ax,
               const uint8_t* ay, const uint8_t* hm, size_t plane, uint8_t* ok, bjj::U128* table,
               const bjj::CombEntry* comb, int mode, unsigned long long* work);
void verify_exact(int grid, cudaStream_t st, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s, const uint8_t* ax,
                  const uint8_t* ay, const uint8_t* hm, uint8_t* ok, bjj::ExactQueue qa, bjj::ExactQueue qr,
                  const bjj::CombEntry* comb, int mode, unsigned long long* work);
void mul_scalar(int grid, cudaStream_t st, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* k,
                bjj::ProjScratch scr, bjj::U128* table, bjj::ExactQueue q, uint32_t* gflags);
void mul_scalar_exact(int grid, cudaStream_t st, const uint8_t* px, const uint8_t* py, const uint8_t* k, int k_words, uint8_t* rx,
                      uint8_t* ry, bjj::ExactQueue q);
void reduce_scalars(int grid, cudaStream_t st, size_t n, const uint8_t* wide, int k_words, uint8_t* out32);
void sign(int grid, cudaStream_t st, size_t n, const uint8_t* key, const uint8_t* msg, uint8_t* r8x, uint8_t* r8y,
          uint8_t* s32, uint8_t* status, const bjj::CombEntry* comb);
void sign_scalars(int grid, cudaStream_t st, size_t n, const uint8_t* key, const uint8_t* msg, uint8_t* sk, uint8_t* r, uint8_t* msgc,
                  uint8_t* status);
void sign_finish(int grid, cudaStream_t st, size_t n, const uint8_t* hm, const uint8_t* sk, const uint8_t* r, const uint8_t* status,
                 uint8_t* r8x, uint8_t* r8y, uint8_t* s32);
void sign_finish_compressed(int grid, cudaStream_t st, size_t n, const uint8_t* hm, const uint8_t* sk, const uint8_t* r,
                            const uint8_t* status, const uint8_t* r8x, const uint8_t* r8y, uint8_t* sig64);
void poseidon(int t, int grid, cudaStream_t st, size_t n, PoseidonIn in, uint8_t* out, uint32_t* gflags);

}  // namespace bjjk
