// sign_batch kernel (reference: PrivateKey::sign, src/lib.rs:308-342).
#include "kernels.h"

using namespace bjj;

__global__ void __launch_bounds__(BJJ_BLOCK, 2) k_sign(size_t n, const uint8_t* key, const uint8_t* msg, uint8_t* r8x,
                                                    uint8_t* r8y, uint8_t* s32, uint8_t* status, const CombEntry* comb) {
    BJJ_LANE_LOOP(n) lane_sign(key, msg, r8x, r8y, s32, status, i, comb);
}

// pipeline flavour: BLAKE-512 twice (ALU only, small) and the final scalar arithmetic; the point and hash work in between
// runs on k_fixed_base / k_batch_affine / k_poseidon<6>
__global__ void __launch_bounds__(BJJ_BLOCK) k_sign_scalars(size_t n, const uint8_t* key, const uint8_t* msg, uint8_t* sk, uint8_t* r,
                                                          uint8_t* msgc, uint8_t* status) {
    BJJ_LANE_LOOP(n) lane_sign_scalars(key, msg, sk, r, msgc, status, i);
}
__global__ void __launch_bounds__(BJJ_BLOCK) k_sign_finish(size_t n, const uint8_t* hm, const uint8_t* sk, const uint8_t* r,
                                                         const uint8_t* status, uint8_t* r8x, uint8_t* r8y, uint8_t* s32) {
    BJJ_LANE_LOOP(n) lane_sign_finish(hm, sk, r, status, r8x, r8y, s32, i);
}
// the same last phase writing Signature::compress: compress(R8) || S into lane i of sig64 (64-byte stride)
__global__ void __launch_bounds__(BJJ_BLOCK) k_sign_finish_compressed(size_t n, const uint8_t* hm, const uint8_t* sk, const uint8_t* r,
                                                                    const uint8_t* status, const uint8_t* r8x, const uint8_t* r8y,
                                                                    uint8_t* sig64) {
    BJJ_LANE_LOOP(n) lane_sign_finish(hm, sk, r, status, SignCompressedOut{r8x, r8y, sig64}, i);
}

// sign_schnorr pipeline (reference: PrivateKey::sign_schnorr, src/lib.rs:344-362, with caller nonces): the scalars
// (BLAKE-512 once, the nonce mod SUBORDER) and the exact s = k + sk * h; r, pk and h run on k_fixed_base /
// k_batch_affine / k_poseidon<6> in between
__global__ void __launch_bounds__(BJJ_BLOCK) k_sign_schnorr_scalars(size_t n, const uint8_t* key, const uint8_t* msg,
                                                                  const uint8_t* nonce, int nonce_words, uint8_t* sk, uint8_t* kr,
                                                                  uint8_t* msgc, uint8_t* status) {
    BJJ_LANE_LOOP(n) lane_sign_schnorr_scalars(key, msg, nonce, nonce_words, sk, kr, msgc, status, i);
}
__global__ void __launch_bounds__(BJJ_BLOCK) k_sign_schnorr_finish(size_t n, const uint8_t* h, const uint8_t* sk, const uint8_t* nonce,
                                                                 int nonce_words, const uint8_t* status, uint8_t* rx, uint8_t* ry,
                                                                 uint8_t* s) {
    BJJ_LANE_LOOP(n) lane_sign_schnorr_finish(h, sk, nonce, nonce_words, status, rx, ry, s, i);
}

namespace bjjk {

void sign_schnorr_scalars(int grid, cudaStream_t st, size_t n, const uint8_t* key, const uint8_t* msg, const uint8_t* nonce,
                          int nonce_words, uint8_t* sk, uint8_t* kr, uint8_t* msgc, uint8_t* status) {
    k_sign_schnorr_scalars<<<grid, BJJ_BLOCK, 0, st>>>(n, key, msg, nonce, nonce_words, sk, kr, msgc, status);
}
void sign_schnorr_finish(int grid, cudaStream_t st, size_t n, const uint8_t* h, const uint8_t* sk, const uint8_t* nonce, int nonce_words,
                         const uint8_t* status, uint8_t* rx, uint8_t* ry, uint8_t* s) {
    k_sign_schnorr_finish<<<grid, BJJ_BLOCK, 0, st>>>(n, h, sk, nonce, nonce_words, status, rx, ry, s);
}

int sign_blocks_per_sm() { return blocks_per_sm(k_sign); }
void sign(int grid, cudaStream_t st, size_t n, const uint8_t* key, const uint8_t* msg, uint8_t* r8x, uint8_t* r8y,
          uint8_t* s32, uint8_t* status, const CombEntry* comb) {
    k_sign<<<grid, BJJ_BLOCK, 0, st>>>(n, key, msg, r8x, r8y, s32, status, comb);
}

void sign_scalars(int grid, cudaStream_t st, size_t n, const uint8_t* key, const uint8_t* msg, uint8_t* sk, uint8_t* r, uint8_t* msgc,
                  uint8_t* status) {
    k_sign_scalars<<<grid, BJJ_BLOCK, 0, st>>>(n, key, msg, sk, r, msgc, status);
}
void sign_finish(int grid, cudaStream_t st, size_t n, const uint8_t* hm, const uint8_t* sk, const uint8_t* r, const uint8_t* status,
                 uint8_t* r8x, uint8_t* r8y, uint8_t* s32) {
    k_sign_finish<<<grid, BJJ_BLOCK, 0, st>>>(n, hm, sk, r, status, r8x, r8y, s32);
}
void sign_finish_compressed(int grid, cudaStream_t st, size_t n, const uint8_t* hm, const uint8_t* sk, const uint8_t* r,
                            const uint8_t* status, const uint8_t* r8x, const uint8_t* r8y, uint8_t* sig64) {
    k_sign_finish_compressed<<<grid, BJJ_BLOCK, 0, st>>>(n, hm, sk, r, status, r8x, r8y, sig64);
}

}  // namespace bjjk
