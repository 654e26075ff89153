// poseidon_batch kernels, t = 2..7 (reference: POSEIDON.hash, poseidon-rs 0.0.8 behind src/lib.rs:59; that crate's hash()
// rejects an empty input and more than 6 inputs -- `inp.len() >= n_rounds_p.len() - 1` with its 8-entry round table).
#include "kernels.h"

using namespace bjj;

template <int T>
__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_poseidon(size_t n, PoseidonIn in, uint8_t* out, uint32_t* gflags) {
    BJJ_FLAGS_BEGIN
    BJJ_LANE_LOOP(n) lane_poseidon<T>(in.p, out, i, flags);
    BJJ_FLAGS_END(gflags)
}

namespace bjjk {

int poseidon_blocks_per_sm(int t) {
    switch (t) {
        case 2: return blocks_per_sm(k_poseidon<2>);
        case 3: return blocks_per_sm(k_poseidon<3>);
        case 4: return blocks_per_sm(k_poseidon<4>);
        case 5: return blocks_per_sm(k_poseidon<5>);
        case 6: return blocks_per_sm(k_poseidon<6>);
        default: return blocks_per_sm(k_poseidon<7>);
    }
}

void poseidon(int t, int grid, cudaStream_t st, size_t n, PoseidonIn in, uint8_t* out, uint32_t* gflags) {
    switch (t) {
        case 2: k_poseidon<2><<<grid, BJJ_BLOCK, 0, st>>>(n, in, out, gflags); break;
        case 3: k_poseidon<3><<<grid, BJJ_BLOCK, 0, st>>>(n, in, out, gflags); break;
        case 4: k_poseidon<4><<<grid, BJJ_BLOCK, 0, st>>>(n, in, out, gflags); break;
        case 5: k_poseidon<5><<<grid, BJJ_BLOCK, 0, st>>>(n, in, out, gflags); break;
        case 6: k_poseidon<6><<<grid, BJJ_BLOCK, 0, st>>>(n, in, out, gflags); break;
        default: k_poseidon<7><<<grid, BJJ_BLOCK, 0, st>>>(n, in, out, gflags); break;
    }
}

}  // namespace bjjk
