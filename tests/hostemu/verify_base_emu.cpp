// TEST HARNESS ONLY -- never shipped, never loaded by the product.
//
// The lane bodies of verify_base (lanes.cuh: lane_verify_base_hash, lane_verify_base_ec, and the R8 phases of
// decompression) compiled for the HOST with BJJ_HOST_EMU, as hostemu.cpp does for the other lane bodies.
// tests/test_verify_base.py builds it and checks it against the oracle's verify without a GPU.
#define BJJ_HOST_EMU 1
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../babyjubjub-rs_b200/csrc/lanes.cuh"

using namespace bjj;

// two tables filled on demand: B8's and the key's (the device builds all entries in k_comb_build / k_comb_build_point)
struct EmuComb {
    CombEntry* comb = nullptr;
    uint8_t* valid = nullptr;
    bool is_b8 = true;
    PointAff p;
    void init() {
        if (!comb) {
            comb = (CombEntry*)calloc(BJJ_COMB_TOTAL, sizeof(CombEntry));     // pages are committed on first touch
            valid = (uint8_t*)calloc(BJJ_COMB_TOTAL, 1);
        }
    }
};
static EmuComb g_b8, g_key;

namespace bjj {
void bjj_emu_need_comb_entry(const CombEntry* comb, int w, int j) {
    EmuComb* c = comb == g_b8.comb ? &g_b8 : comb == g_key.comb ? &g_key : nullptr;
    const size_t idx = (size_t)w * BJJ_COMB_ENTRIES + j;
    if (!c || c->valid[idx]) return;
    c->valid[idx] = 1;
    if (c->is_b8)
        comb_build_entry(c->comb, w, j);
    else
        comb_build_entry(c->comb, w, j, c->p);
}
}  // namespace bjj

// selects the key (canonical little-endian coordinates of an on-curve point); its table starts empty
static void set_key(const uint8_t* ax32, const uint8_t* ay32, PointAff& a) {
    g_b8.init();
    g_key.init();
    uint32_t flags = 0;
    load_fr(a.x, ax32, 0, flags);
    load_fr(a.y, ay32, 0, flags);
    g_key.is_b8 = false;
    g_key.p = a;
    memset(g_key.valid, 0, BJJ_COMB_TOTAL);
}

extern "C" {

// bjj_verify_base_batch as its two kernels run it; returns the NONCANONICAL flag bits
uint32_t emu_verify_base(size_t n, const uint8_t* ax32, const uint8_t* ay32, const uint8_t* r8x, const uint8_t* r8y,
                         const uint8_t* s32, const uint8_t* msg32, uint8_t* ok) {
    PointAff a;
    set_key(ax32, ay32, a);
    std::vector<uint8_t> hm(32 * (n + 1));
    uint32_t flags = 0;
    for (size_t i = 0; i < n; i++) lane_verify_base_hash(r8x, r8y, a, msg32, nullptr, hm.data(), ok, i, flags);
    for (size_t i = 0; i < n; i++) lane_verify_base_ec(r8x, r8y, s32, 1, 0, hm.data(), ok, i, g_b8.comb, g_key.comb);
    return flags;
}

// bjj_verify_base_compressed_batch: R8 decompressed in three phases (one shared inversion), then the two kernels
void emu_verify_base_compressed(size_t n, const uint8_t* ax32, const uint8_t* ay32, const uint8_t* sig64, const uint8_t* msg32,
                                uint8_t* ok, uint8_t* status) {
    PointAff a;
    set_key(ax32, ay32, a);
    std::vector<uint8_t> buf(32 * 7 * (n + 1));
    uint8_t *hm = buf.data(), *dx = hm + 32 * n, *dy = dx + 32 * n;
    ProjScratch scr;
    scr.x = dy + 32 * n;
    scr.y = scr.x + 32 * n;
    scr.z = scr.y + 32 * n;
    scr.p = scr.z + 32 * n;
    for (size_t i = 0; i < n; i++) lane_decompress_prepare(sig64, 2, 0, scr, i, i);
    for (size_t t = 0; t < 3; t++) batch_inverse_strided(scr, n, t, 3);
    for (size_t i = 0; i < n; i++) lane_decompress_finish(sig64, 2, 0, scr, i, dx, dy, status, i, false);
    uint32_t flags = 0;
    for (size_t i = 0; i < n; i++) lane_verify_base_hash(dx, dy, a, msg32, status, hm, ok, i, flags);
    for (size_t i = 0; i < n; i++) lane_verify_base_ec(dx, dy, sig64, 2, 1, hm, ok, i, g_b8.comb, g_key.comb);
}

// k = 8*hm mod ORDER (the scalar of the key's comb walk)
void emu_verify_base_scalar(size_t n, const uint8_t* hm32, uint8_t* k32) {
    for (size_t i = 0; i < n; i++) {
        uint32_t hm[8], k[8];
        load_u256(hm, hm32, i);
        verify_base_scalar(k, hm);
        store_u256(k32, i, k);
    }
}

}  // extern "C"
