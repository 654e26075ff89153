// TEST HARNESS ONLY -- never shipped, never loaded by the product.
//
// The Schnorr signing lane bodies of the device code (lanes.cuh: lane_sign_schnorr_scalars, lane_sign_schnorr_finish
// and lane_mod_suborder_wide) compiled for the HOST with BJJ_HOST_EMU, in the order of bjj_cuda.cu::launch_sign_schnorr.
// tests/test_sign_schnorr.py builds it and checks it against the oracle without a GPU.
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

// B8 * k for the 256-bit scalars k of n lanes: the fixed-base lanes, then the batched affine pass with 3 "threads"
static void fixed_base(const uint8_t* k, uint8_t* rx, uint8_t* ry, size_t n) {
    std::vector<uint8_t> scr_buf(4 * 32 * (n + 1), 0);
    ProjScratch scr;
    scr.x = scr_buf.data();
    scr.y = scr.x + 32 * n;
    scr.z = scr.y + 32 * n;
    scr.p = scr.z + 32 * n;
    for (size_t i = 0; i < n; i++) lane_fixed_base(k, scr, i, g_comb);
    const size_t T = 3;
    for (size_t t = 0; t < T; t++) batch_affine_strided(scr, AffineOut{rx, ry}, n, t, T);
}

extern "C" {

// wide mod SUBORDER (nwords words per lane) -> 32 bytes per lane
void emu_mod_suborder_wide(size_t n, const uint8_t* wide, int nwords, uint8_t* out32) {
    for (size_t i = 0; i < n; i++) {
        uint32_t acc[8];
        lane_mod_suborder_wide(acc, wide, nwords, i);
        store_u256(out32, i, acc);
    }
}

// sign_schnorr(key, msg, k) as the kernel pipeline runs it: scalars -> r = kr * B8 into (rx, ry), pk = sk * B8 ->
// Poseidon(pk, r, msg) -> the finish (s: nwords + 8 words per lane)
void emu_sign_schnorr(size_t n, const uint8_t* key, const uint8_t* msg, const uint8_t* nonce, int nwords, uint8_t* rx, uint8_t* ry,
                      uint8_t* s, uint8_t* status) {
    init_comb();
    std::vector<uint8_t> buf(6 * 32 * (n + 1));
    uint8_t *sk = buf.data(), *kr = sk + 32 * n, *msgc = kr + 32 * n, *h = msgc + 32 * n, *pkx = h + 32 * n, *pky = pkx + 32 * n;
    for (size_t i = 0; i < n; i++) lane_sign_schnorr_scalars(key, msg, nonce, nwords, sk, kr, msgc, status, i);
    fixed_base(kr, rx, ry, n);
    fixed_base(sk, pkx, pky, n);
    const uint8_t* ins[5] = {pkx, pky, rx, ry, msgc};
    uint32_t flags = 0;
    for (size_t i = 0; i < n; i++) lane_poseidon<6>(ins, h, i, flags);
    for (size_t i = 0; i < n; i++) lane_sign_schnorr_finish(h, sk, nonce, nwords, status, rx, ry, s, i);
}

}  // extern "C"
