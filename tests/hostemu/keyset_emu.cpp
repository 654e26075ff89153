// TEST HARNESS ONLY -- never shipped, never loaded by the product.
//
// The key-set lane bodies (lanes.cuh: recode8, lane_keyset_check / lane_keyset_build + the batched affine pass into
// the compact tables, lane_keyset_mul, lane_verify_keyset_hash / lane_verify_keyset_ec) compiled for the HOST with
// BJJ_HOST_EMU, as verify_base_emu.cpp does for verify_base.  tests/test_verify_keyset.py builds it and checks it
// against the oracle without a GPU.  The compact tables are built whole (4,130 entries per key); B8's 16-bit table is
// filled on demand.
#define BJJ_HOST_EMU 1
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../babyjubjub-rs_b200/csrc/lanes.cuh"

using namespace bjj;

static CombEntry* g_b8 = nullptr;
static uint8_t* g_b8_valid = nullptr;

namespace bjj {
void bjj_emu_need_comb_entry(const CombEntry* comb, int w, int j) {
    const size_t idx = (size_t)w * BJJ_COMB_ENTRIES + j;
    if (comb != g_b8 || g_b8_valid[idx]) return;
    g_b8_valid[idx] = 1;
    comb_build_entry(g_b8, w, j);
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

// the 32 digits and the carry of recode8 for each scalar: digits (n x 33 int32), digit 32 = the carry
void emu_recode8(size_t n, const uint8_t* k32, int32_t* digits) {
    for (size_t i = 0; i < n; i++) {
        uint32_t k[8];
        load_u256(k, k32, i);
        Recode8 rc;
        recode8(rc, k);
        for (int d = 0; d < 32; d++) digits[33 * i + d] = recode8_digit(rc, d);
        digits[33 * i + 32] = (int32_t)rc.top;
    }
}

// bjj_keyset_create's check and build, with the kernels' lane bodies; returns 0 and keeps the set, or the BJJ_BASE_*
// code of the first bad key (status: one code per key)
uint32_t emu_keyset_create(size_t n, const uint8_t* ax, const uint8_t* ay, uint8_t* status) {
    if (!g_b8) {
        g_b8 = (CombEntry*)calloc(BJJ_COMB_TOTAL, sizeof(CombEntry));
        g_b8_valid = (uint8_t*)calloc(BJJ_COMB_TOTAL, 1);
    }
    g_ks.n = n;
    g_ks.keys.assign(64 * n, 0);
    memcpy(g_ks.keys.data(), ax, 32 * n);
    memcpy(g_ks.keys.data() + 32 * n, ay, 32 * n);
    uint8_t *kx = g_ks.keys.data(), *ky = kx + 32 * n;
    uint32_t bad = 0;
    for (size_t i = 0; i < n; i++) {
        status[i] = (uint8_t)lane_keyset_check(kx, ky, i);
        if (status[i] && !bad) bad = status[i];
    }
    if (bad) return bad;
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

// entry (w, j) of key `key` back on the original curve: canonical (x, y); returns 1 iff its t2d = 2d'xy holds
uint32_t emu_keyset_entry(size_t key, int w, int j, uint8_t* x32, uint8_t* y32) {
    const CombEntry& e = g_ks.tables[key * BJJ_KEY_COMB_TOTAL + (size_t)w * Comb8::ENTRIES + j];
    Fr ypx, ymx, t2d, xe, y, two, half, x, t;
    fr_set(ypx, e.ypx);
    fr_set(ymx, e.ymx);
    fr_set(t2d, e.t2d);
    two = fr_const(BJJ_ONE_M);
    fr_dbl(two, two);
    fr_inv(half, two);
    fr_sub(xe, ypx, ymx);
    fr_mul(xe, xe, half);
    fr_add(y, ypx, ymx);
    fr_mul(y, y, half);
    fr_mul(t, xe, y);
    const Fr d2 = fr_const(BJJ_TWO_DP_M);
    fr_mul(t, t, d2);
    const Fr si = fr_const(BJJ_INV_SQRT_NEG_A_M);
    fr_mul(x, xe, si);
    store_fr(x32, 0, x);
    store_fr(y32, 0, y);
    return fr_eq(t, t2d) ? 1u : 0u;
}

// bjj_keyset_mul_batch: lane_keyset_mul then the batched affine pass; returns the flag bits
uint32_t emu_keyset_mul(size_t n, const uint8_t* key_index, const uint8_t* k32, uint8_t* rx, uint8_t* ry) {
    std::vector<uint8_t> buf(128 * (n + 1));
    ProjScratch scr;
    scr.x = buf.data();
    scr.y = scr.x + 32 * n;
    scr.z = scr.y + 32 * n;
    scr.p = scr.z + 32 * n;
    uint32_t flags = 0;
    for (size_t i = 0; i < n; i++) lane_keyset_mul(k32, key_index, (uint32_t)g_ks.n, g_ks.tables.data(), scr, i, flags);
    for (size_t t = 0; t < 3; t++) batch_affine_strided(scr, rx, ry, n, t, 3);
    return flags;
}

// bjj_verify_keyset_batch as its two kernels run it; returns the flag bits
uint32_t emu_verify_keyset(size_t n, const uint8_t* key_index, const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32,
                           const uint8_t* msg32, uint8_t* ok) {
    const uint8_t *kx = g_ks.keys.data(), *ky = kx + 32 * g_ks.n;
    std::vector<uint8_t> hm(32 * (n + 1));
    uint32_t flags = 0;
    for (size_t i = 0; i < n; i++)
        lane_verify_keyset_hash(r8x, r8y, key_index, kx, ky, (uint32_t)g_ks.n, msg32, nullptr, hm.data(), ok, i, flags);
    for (size_t i = 0; i < n; i++)
        lane_verify_keyset_ec(r8x, r8y, s32, 1, 0, hm.data(), ok, i, g_b8, key_index, (uint32_t)g_ks.n, g_ks.tables.data());
    return flags;
}

// bjj_verify_keyset_compressed_batch: R8 decompressed in three phases, then the two kernels; returns the flag bits
uint32_t emu_verify_keyset_compressed(size_t n, const uint8_t* key_index, const uint8_t* sig64, const uint8_t* msg32, uint8_t* ok,
                                      uint8_t* status) {
    const uint8_t *kx = g_ks.keys.data(), *ky = kx + 32 * g_ks.n;
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
    for (size_t i = 0; i < n; i++)
        lane_verify_keyset_hash(dx, dy, key_index, kx, ky, (uint32_t)g_ks.n, msg32, status, hm, ok, i, flags);
    for (size_t i = 0; i < n; i++)
        lane_verify_keyset_ec(dx, dy, sig64, 2, 1, hm, ok, i, g_b8, key_index, (uint32_t)g_ks.n, g_ks.tables.data());
    return flags;
}

}  // extern "C"
