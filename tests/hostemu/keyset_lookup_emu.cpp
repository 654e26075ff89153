// TEST HARNESS ONLY -- never shipped, never loaded by the product.
//
// The key-set index by compressed bytes (lanes.cuh: keyset_index_build, as bjj_keyset_create runs it on the host, and
// the lane body lane_keyset_lookup of k_keyset_lookup) compiled for the HOST with BJJ_HOST_EMU.  The seed is the
// caller's, so that tests/test_keyset_lookup.py can fix it and craft keys that share a probe chain.
#define BJJ_HOST_EMU 1
#include <stdlib.h>
#include <string.h>
#include <vector>
#include "../../babyjubjub-rs_b200/csrc/lanes.cuh"

using namespace bjj;

static std::vector<uint8_t> g_comp;
static std::vector<uint32_t> g_slots;
static uint64_t g_seed = 0;

extern "C" {

// builds the index of n keys (canonical affine coordinates, 32 B each) under `seed`; returns the number of slots
size_t emu_lookup_build(size_t n, const uint8_t* ax, const uint8_t* ay, uint64_t seed) {
    g_seed = seed;
    g_comp.assign(32 * n, 0);
    g_slots.assign(keyset_index_slots(n), 0);
    keyset_index_build(n, ax, ay, seed, g_comp.data(), g_slots.data());
    return g_slots.size();
}

// the built table: slots (one key index or BJJ_KEY_NONE each) and the compressed keys (32 B per key)
void emu_lookup_table(uint32_t* slots, uint8_t* comp) {
    memcpy(slots, g_slots.data(), 4 * g_slots.size());
    memcpy(comp, g_comp.data(), g_comp.size());
}

// keyset_hash of each 32-byte lane under `seed`
void emu_lookup_hash(size_t n, const uint8_t* pk32, uint64_t seed, uint64_t* out) {
    for (size_t i = 0; i < n; i++) {
        uint32_t b[8];
        load_u256(b, pk32, i);
        out[i] = keyset_hash(b, seed);
    }
}

// lane_keyset_lookup of every lane against the built index
void emu_lookup(size_t n, const uint8_t* pk32, uint32_t* key_index) {
    for (size_t i = 0; i < n; i++)
        lane_keyset_lookup(pk32, g_comp.data(), g_slots.data(), g_slots.size() - 1, g_seed, key_index, i);
}

}  // extern "C"
