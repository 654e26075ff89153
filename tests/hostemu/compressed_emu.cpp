// TEST HARNESS ONLY -- never shipped, never loaded by the product.
//
// The compressed output forms of the device code (lanes.cuh: batch_affine_strided with CompressedOut,
// lane_sign_finish with SignCompressedOut) compiled for the HOST with BJJ_HOST_EMU, as hostemu.cpp does for the
// other lane bodies.  tests/test_compressed_outputs.py builds it and checks it against the oracle without a GPU.
#define BJJ_HOST_EMU 1
#include <stdlib.h>
#include <vector>
#include "../../babyjubjub-rs_b200/csrc/lanes.cuh"

using namespace bjj;

static CombEntry* g_comb = nullptr;
static uint8_t* g_comb_valid = nullptr;

// comb entries are built on demand (the device builds all of them in k_comb_build; here a test touches a few)
namespace bjj {
void bjj_emu_need_comb_entry(const CombEntry* comb, int w, int j) {
    const size_t idx = (size_t)w * BJJ_COMB_ENTRIES + j;
    if (comb != g_comb || g_comb_valid[idx]) return;
    g_comb_valid[idx] = 1;
    comb_build_entry(g_comb, w, j);
}
}  // namespace bjj

static void init_comb() {
    if (g_comb) return;
    g_comb = (CombEntry*)calloc(BJJ_COMB_TOTAL, sizeof(CombEntry));     // pages are committed on first touch
    g_comb_valid = (uint8_t*)calloc(BJJ_COMB_TOTAL, 1);
}

static std::vector<uint8_t> g_scr;
static ProjScratch proj_scratch(size_t n) {
    g_scr.assign(4 * 32 * (n + 1), 0);
    ProjScratch s;
    s.x = g_scr.data();
    s.y = s.x + 32 * n;
    s.z = s.y + 32 * n;
    s.p = s.z + 32 * n;
    return s;
}

// the batched affine pass in output form `out` with T "threads" (T = 3 exercises several strides and ragged tails)
template <class Out>
static void batch_affine(const ProjScratch& s, Out out, size_t n) {
    const size_t T = 3;
    for (size_t t = 0; t < T; t++) batch_affine_strided(s, out, n, t, T);
}

extern "C" {

// compress(public(key)): the public-key lanes, then the batched affine pass in its compressed form
void emu_public_compressed(size_t n, const uint8_t* key, uint8_t* out32) {
    init_comb();
    ProjScratch scr = proj_scratch(n);
    for (size_t i = 0; i < n; i++) lane_public(key, scr, i, g_comb);
    batch_affine(scr, CompressedOut{out32}, n);
}

// sign(key, msg).compress() as the kernel pipeline runs it (bjj_cuda.cu::launch_sign, compressed form): scalars ->
// R8 and A on the fixed-base path -> Poseidon(R8, A, msg) -> the compressed finish
void emu_sign_compressed(size_t n, const uint8_t* key, const uint8_t* msg, uint8_t* sig64, uint8_t* status) {
    init_comb();
    std::vector<uint8_t> buf(8 * 32 * (n + 1));
    uint8_t *sk = buf.data(), *r = sk + 32 * n, *msgc = r + 32 * n, *hm = msgc + 32 * n;
    uint8_t *rx = hm + 32 * n, *ry = rx + 32 * n, *ax = ry + 32 * n, *ay = ax + 32 * n;
    for (size_t i = 0; i < n; i++) lane_sign_scalars(key, msg, sk, r, msgc, status, i);
    ProjScratch scr = proj_scratch(n);
    for (size_t i = 0; i < n; i++) lane_fixed_base(r, scr, i, g_comb);
    batch_affine(scr, AffineOut{rx, ry}, n);
    scr = proj_scratch(n);
    for (size_t i = 0; i < n; i++) lane_fixed_base(sk, scr, i, g_comb);
    batch_affine(scr, AffineOut{ax, ay}, n);
    const uint8_t* ins[5] = {rx, ry, ax, ay, msgc};
    uint32_t flags = 0;
    for (size_t i = 0; i < n; i++) lane_poseidon<6>(ins, hm, i, flags);
    for (size_t i = 0; i < n; i++) lane_sign_finish(hm, sk, r, status, SignCompressedOut{rx, ry, sig64}, i);
}

}  // extern "C"
