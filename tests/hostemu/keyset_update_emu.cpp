// TEST HARNESS ONLY -- never shipped, never loaded by the product.
//
// The index side of bjj_keyset_append / bjj_keyset_replace compiled for the HOST with BJJ_HOST_EMU: the set's host copy
// of the compressed keys is edited with keyset_compress and the slots are rebuilt from it with keyset_index_fill, as
// keyset_edit (bjj_cuda.cu) does, then lane_keyset_lookup runs against the result.
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

// an empty set under `seed`
void emu_update_reset(uint64_t seed) {
    g_seed = seed;
    g_comp.clear();
    g_slots.clear();
}

// keys first .. first + n - 1 get the coordinates ax, ay (first == the set's size appends them); returns the new size
size_t emu_update_edit(size_t first, size_t n, const uint8_t* ax, const uint8_t* ay) {
    const size_t n1 = first + n > g_comp.size() / 32 ? first + n : g_comp.size() / 32;
    g_comp.resize(32 * n1);
    for (size_t j = 0; j < n; j++) keyset_compress(ax, ay, j, g_comp.data() + 32 * (first + j));
    g_slots.assign(keyset_index_slots(n1), 0);
    keyset_index_fill(n1, g_comp.data(), g_seed, g_slots.data());
    return n1;
}

// the slot count and the compressed keys (32 B per key)
size_t emu_update_table(uint8_t* comp) {
    memcpy(comp, g_comp.data(), g_comp.size());
    return g_slots.size();
}

// lane_keyset_lookup of every lane against the current index
void emu_update_lookup(size_t n, const uint8_t* pk32, uint32_t* key_index) {
    for (size_t i = 0; i < n; i++)
        lane_keyset_lookup(pk32, g_comp.data(), g_slots.data(), g_slots.size() - 1, g_seed, key_index, i);
}

// keyset_indexed of each 32-byte lane
void emu_update_indexed(size_t n, const uint8_t* c, uint8_t* out) {
    for (size_t i = 0; i < n; i++) out[i] = keyset_indexed(c + 32 * i) ? 1 : 0;
}

}  // extern "C"
