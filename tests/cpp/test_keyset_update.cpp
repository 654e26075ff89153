// KeySet::append and KeySet::replace of the C++ host mirror (host/bjj.hpp): lookups and verify on the edited set equal
// those of a set created from the same key list, and a refused edit (an off-curve key, a range past the set) leaves the
// set as it was.  Built by tests/test_keyset_update.py; runs on the GPU box (`-m gpu`).  Exit code 0 = all passed.
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
        for (int i = 0; i < 32; i++) keys[k].key[i] = (uint8_t)(i % 11 + 19 * k);
    std::vector<Point> pks;
    std::vector<std::array<uint8_t, 32>> comp;
    for (const PrivateKey& k : keys) {
        pks.push_back(k.public_key());
        comp.push_back(pks.back().compress());
    }
    KeySet ks({pks[0], pks[1], pks[2]});
    ks.append({pks[1], pks[3]});                        // key 1 twice: found at 1
    CHECK(ks.size() == 5);
    CHECK(ks.lookup(comp) == std::vector<uint32_t>({0, 1, 2, 4}));
    ks.replace(1, {pks[3]});                            // key 1's old bytes are now found at its duplicate, 3
    CHECK(ks.size() == 5);
    CHECK(ks.lookup(comp) == std::vector<uint32_t>({0, 3, 2, 1}));

    Point off = pks[0];
    off.x[0] ^= 1;                                      // off the curve
    std::vector<uint8_t> st;
    bool threw = false;
    try {
        ks.append({pks[2], off}, &st);
    } catch (const Error& e) {
        threw = e.code == BJJ_ERR_ARG;
    }
    CHECK(threw && st == std::vector<uint8_t>({BJJ_KEY_OK, BJJ_KEY_OFF_CURVE}));
    threw = false;
    try {
        ks.replace(4, {pks[0], pks[0]});
    } catch (const Error& e) {
        threw = e.code == BJJ_ERR_ARG;
    }
    CHECK(threw && ks.size() == 5);
    CHECK(ks.lookup(comp) == std::vector<uint32_t>({0, 3, 2, 1}));

    // the current list is {0, 3, 2, 1, 3}: verify on the edited set equals verify on a set created from that list
    KeySet fresh({pks[0], pks[3], pks[2], pks[1], pks[3]});
    const std::vector<uint32_t> who = {0, 3, 2, 1, 3, 1};
    const std::vector<uint32_t> priv = {0, 1, 2, 3, 1, 0};    // the key each index holds; the last lane names key 3 but is signed by key 0
    std::vector<Signature> sigs;
    std::vector<U256> msgs;
    for (size_t i = 0; i < who.size(); i++) {
        msgs.push_back(u256_from_u64(500 + i));
        sigs.push_back(keys[priv[i]].sign(msgs.back()));
    }
    const std::vector<uint8_t> ok = ks.verify_batch(who, sigs, msgs);
    CHECK(ok == std::vector<uint8_t>({1, 1, 1, 1, 1, 0}));
    CHECK(ok == fresh.verify_batch(who, sigs, msgs));
    std::printf("keyset update ok\n");
    return 0;
}
