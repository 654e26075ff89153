// KeySet::lookup and KeySet::verify_compressed_by_key of the C++ host mirror (host/bjj.hpp) against
// verify_compressed_batch and KeySet::verify_compressed_batch with the found indices.  Built by
// tests/test_keyset_lookup.py; runs on the GPU box (`-m gpu`).  Exit code 0 = all passed.
#include <cstdio>

#include "../../host/bjj.hpp"

using namespace bjj_host;

#define CHECK(c)                                                                  \
    do {                                                                          \
        if (!(c)) {                                                               \
            std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #c);   \
            return 1;                                                             \
        }                                                                         \
    } while (0)

int main() {
    std::vector<PrivateKey> keys(4);
    for (int k = 0; k < 4; k++)
        for (int i = 0; i < 32; i++) keys[k].key[i] = (uint8_t)(i % 10 + 17 * k);
    std::vector<Point> pks;
    for (const PrivateKey& k : keys) pks.push_back(k.public_key());
    // the set holds keys 0..2 and key 1 twice; key 3 is not in it
    KeySet ks({pks[0], pks[1], pks[2], pks[1]});
    std::vector<std::array<uint8_t, 32>> comp;
    for (const Point& p : pks) comp.push_back(p.compress());
    std::array<uint8_t, 32> flipped = comp[2];
    flipped[31] ^= 0x80;                                // -P_2: not in the set
    auto found = ks.lookup({comp[0], comp[1], comp[2], comp[3], flipped});
    const std::vector<uint32_t> fexpect = {0, 1, 2, BJJ_KEY_NONE, BJJ_KEY_NONE};
    CHECK(found == fexpect);

    const std::vector<uint32_t> who = {0, 1, 2, 3, 1, 0};
    std::vector<std::array<uint8_t, 32>> lane_pk;
    std::vector<std::array<uint8_t, 64>> sigs;
    std::vector<U256> msgs;
    for (size_t i = 0; i < who.size(); i++) {
        msgs.push_back(u256_from_u64(1000 + i));
        sigs.push_back(keys[who[i]].sign(msgs.back()).compress());
        lane_pk.push_back(comp[who[i]]);
    }
    sigs[4][40] ^= 1;                                   // corrupted S
    for (int b = 0; b < 32; b++) sigs[5][b] = 0xff;     // R8 y >= Q
    std::vector<uint8_t> st;
    std::vector<uint32_t> ki;
    auto ok = ks.verify_compressed_by_key(lane_pk, sigs, msgs, &st, &ki);
    const std::vector<uint8_t> okexpect = {1, 1, 1, 0, 0, 0}, stexpect = {0, 0, 0, 0, 0, BJJ_STATUS_Y_RANGE};
    const std::vector<uint32_t> kiexpect = {0, 1, 2, BJJ_KEY_NONE, 1, 0};
    CHECK(ok == okexpect);
    CHECK(st == stexpect);
    CHECK(ki == kiexpect);
    std::vector<uint8_t> wst;
    CHECK(ks.verify_compressed_batch({0, 1, 2}, {sigs[0], sigs[1], sigs[2]}, {msgs[0], msgs[1], msgs[2]}, &wst) ==
          std::vector<uint8_t>({1, 1, 1}));
    std::printf("keyset lookup ok\n");
    return 0;
}
