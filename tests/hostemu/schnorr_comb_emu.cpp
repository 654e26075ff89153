// TEST HARNESS ONLY -- never shipped, never loaded by the product.
//
// The verify_schnorr comb lane bodies (lanes.cuh: lane_verify_base_hash / lane_verify_base_ec and lane_verify_keyset_hash /
// lane_verify_keyset_ec with MODE = BJJ_MODE_SCHNORR) compiled for the HOST with BJJ_HOST_EMU, in the order of
// bjj_cuda.cu::launch_verify_base.  tests/test_verify_schnorr_comb.py builds it and checks it against the oracle's
// verify_schnorr without a GPU.  B8's and the one key's 16-bit tables are filled on demand; a key set's compact tables
// are built whole, as keyset_emu.cpp does.
#define BJJ_HOST_EMU 1
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../babyjubjub-rs_b200/csrc/lanes.cuh"

using namespace bjj;

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

// a key set as bjj_keyset_create builds it: Montgomery key planes and the compact tables
struct EmuKeyset {
    size_t n = 0;
    std::vector<uint8_t> keys;
    std::vector<CombEntry> tables;
};
static EmuKeyset g_ks;

extern "C" {

// bjj_keyset_create's check and build; returns 0, or the BJJ_BASE_* code of the first bad key
uint32_t emu_keyset_create(size_t n, const uint8_t* ax, const uint8_t* ay) {
    g_b8.init();
    g_ks.n = n;
    g_ks.keys.assign(64 * n, 0);
    memcpy(g_ks.keys.data(), ax, 32 * n);
    memcpy(g_ks.keys.data() + 32 * n, ay, 32 * n);
    uint8_t *kx = g_ks.keys.data(), *ky = kx + 32 * n;
    for (size_t i = 0; i < n; i++)
        if (const uint32_t st = lane_keyset_check(kx, ky, i)) return st;
    g_ks.tables.assign(n * BJJ_KEY_COMB_TOTAL, CombEntry{});
    const size_t lanes = n * BJJ_KEY_BUILD_POINTS;
    std::vector<uint8_t> buf(128 * lanes);
    ProjScratch scr;
    scr.x = buf.data();
    scr.y = scr.x + 32 * lanes;
    scr.z = scr.y + 32 * lanes;
    scr.p = scr.z + 32 * lanes;
    for (size_t k = 0; k < n; k++)
        for (int w = 0; w < Comb8::WINDOWS; w++)
            lane_keyset_build(kx, ky, k, w, scr, k * BJJ_KEY_BUILD_POINTS, g_ks.tables.data() + k * BJJ_KEY_COMB_TOTAL);
    for (size_t t = 0; t < 7; t++) batch_affine_strided(scr, KeysetCombOut{g_ks.tables.data()}, lanes, t, 7);
    return 0;
}

// bjj_verify_schnorr_base_batch as its two kernels run it, for the on-curve key (pkx, pky); s_red receives the reduced s
// of the lanes that reach the reduction.  Returns the flag bits.
uint32_t emu_verify_schnorr_base(size_t n, const uint8_t* pkx32, const uint8_t* pky32, const uint8_t* msg32, const uint8_t* rx,
                                 const uint8_t* ry, const uint8_t* s, int nwords, uint8_t* ok, uint8_t* status, uint8_t* s_red) {
    g_b8.init();
    g_key.init();
    PointAff a;
    uint32_t flags = 0;
    load_fr(a.x, pkx32, 0, flags);
    load_fr(a.y, pky32, 0, flags);
    g_key.is_b8 = false;
    g_key.p = a;
    memset(g_key.valid, 0, BJJ_COMB_TOTAL);
    std::vector<uint8_t> hm(32 * (n + 1));
    const SchnorrWide sw{s, nwords, s_red, status};
    flags = 0;
    for (size_t i = 0; i < n; i++) lane_verify_base_hash<BJJ_MODE_SCHNORR>(rx, ry, a, msg32, nullptr, hm.data(), ok, i, flags, sw);
    for (size_t i = 0; i < n; i++) lane_verify_base_ec<Comb16, BJJ_MODE_SCHNORR>(rx, ry, s_red, 1, 0, hm.data(), ok, i, g_b8.comb, g_key.comb);
    return flags;
}

// bjj_verify_schnorr_keyset_batch as its two kernels run it, over the set of emu_keyset_create; returns the flag bits
uint32_t emu_verify_schnorr_keyset(size_t n, const uint8_t* key_index, const uint8_t* msg32, const uint8_t* rx, const uint8_t* ry,
                                   const uint8_t* s, int nwords, uint8_t* ok, uint8_t* status, uint8_t* s_red) {
    const uint8_t *kx = g_ks.keys.data(), *ky = kx + 32 * g_ks.n;
    std::vector<uint8_t> hm(32 * (n + 1));
    const SchnorrWide sw{s, nwords, s_red, status};
    uint32_t flags = 0;
    for (size_t i = 0; i < n; i++)
        lane_verify_keyset_hash<BJJ_MODE_SCHNORR>(rx, ry, key_index, kx, ky, (uint32_t)g_ks.n, msg32, nullptr, hm.data(), ok, i, flags, sw);
    for (size_t i = 0; i < n; i++)
        lane_verify_keyset_ec<BJJ_MODE_SCHNORR>(rx, ry, s_red, 1, 0, hm.data(), ok, i, g_b8.comb, key_index, (uint32_t)g_ks.n,
                                                g_ks.tables.data());
    return flags;
}

}  // extern "C"
