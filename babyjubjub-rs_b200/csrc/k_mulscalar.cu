// mul_scalar_batch kernels (reference: Point::mul_scalar, src/lib.rs:149-164).
#include "kernels.h"

using namespace bjj;

// 2 resident CTAs per SM (up to 255 registers): measured 26.1 M mults/s against 21.4 M/s with the
// 168-register cap of 3 CTAs -- the ladder gains more from registers (ILP, no spills) than from warps
#ifndef BJJ_MULSCALAR_MINB
#define BJJ_MULSCALAR_MINB 2
#endif

__global__ void __launch_bounds__(BJJ_BLOCK, BJJ_MULSCALAR_MINB) k_mul_scalar(size_t n, const uint8_t* px, const uint8_t* py,
                                                          const uint8_t* k, ProjScratch scr, U128* table,
                                                          ExactQueue q, uint32_t* gflags) {
    BJJ_FLAGS_BEGIN
    const LaneTable tbl = thread_table(table);
    BJJ_LANE_LOOP(n) lane_mul_scalar(px, py, k, scr, i, tbl, q, flags);
    BJJ_FLAGS_END(gflags)
}

__global__ void __launch_bounds__(BJJ_EXACT_BLOCK) k_mul_scalar_exact(const uint8_t* px, const uint8_t* py, const uint8_t* k, int k_words,
                                                                      uint8_t* rx, uint8_t* ry, ExactQueue q) {
    BJJ_QUEUE_LOOP(q) lane_mul_scalar_exact(px, py, k, k_words, rx, ry, q.list[j]);
}

// wide scalars (more than 256 bits) -> scalar mod ORDER for the fast ladder of the on-curve lanes
__global__ void __launch_bounds__(BJJ_BLOCK) k_reduce_scalars(size_t n, const uint8_t* wide, int k_words, uint8_t* out32) {
    BJJ_LANE_LOOP(n) lane_reduce_scalar_order(wide, k_words, out32, i);
}

namespace bjjk {

int mul_scalar_blocks_per_sm() { return blocks_per_sm(k_mul_scalar); }
void mul_scalar(int grid, cudaStream_t st, size_t n, const uint8_t* px, const uint8_t* py, const uint8_t* k, ProjScratch scr,
                U128* table, ExactQueue q, uint32_t* gflags) {
    k_mul_scalar<<<grid, BJJ_BLOCK, 0, st>>>(n, px, py, k, scr, table, q, gflags);
}
void mul_scalar_exact(int grid, cudaStream_t st, const uint8_t* px, const uint8_t* py, const uint8_t* k, int k_words, uint8_t* rx,
                      uint8_t* ry, ExactQueue q) {
    k_mul_scalar_exact<<<grid, BJJ_EXACT_BLOCK, 0, st>>>(px, py, k, k_words, rx, ry, q);
}
void reduce_scalars(int grid, cudaStream_t st, size_t n, const uint8_t* wide, int k_words, uint8_t* out32) {
    k_reduce_scalars<<<grid, BJJ_BLOCK, 0, st>>>(n, wide, k_words, out32);
}

}  // namespace bjjk
