// public_compressed_batch / sign_compressed_batch of the C++ host mirror (host/bjj.hpp) against the one-lane
// compress() calls.  Built by tests/test_compressed_outputs.py; runs on the GPU box (`-m gpu`).  Exit code 0 = all passed.
#include <cstdio>
#include <cstring>
#include <string>

#include "../../host/bjj.hpp"

using namespace bjj_host;

static U256 from_hex_be(const std::string& h) {
    U256 r{};
    std::string s = h;
    while (s.size() < 64) s = "0" + s;
    for (int i = 0; i < 32; i++) r[31 - i] = (uint8_t)std::stoi(s.substr(2 * i, 2), nullptr, 16);
    return r;
}
#define CHECK(c)                                                                  \
    do {                                                                          \
        if (!(c)) {                                                               \
            std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #c);   \
            return 1;                                                             \
        }                                                                         \
    } while (0)

int main() {
    // the circomlib key of the reference's test vectors (src/lib.rs:688-738), then a few others
    std::vector<PrivateKey> keys;
    for (int k = 0; k < 6; k++) {
        PrivateKey pk;
        for (int i = 0; i < 32; i++) pk.key[i] = k == 0 ? (uint8_t)(i % 10) : (uint8_t)(37 * k + 11 * i);
        keys.push_back(pk);
    }
    const U256 q = from_hex_be("30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001");
    U256 over = q;
    over[0] += 1;                                       // Q + 1: "msg outside the Finite Field"
    std::vector<U256> msgs = {u256_from_u64(0x0908070605040302ull), u256_from_u64(0), u256_from_u64(1), q, over,
                              from_hex_be("1234567890abcdef")};

    auto pubs = public_compressed_batch(keys);
    CHECK(pubs.size() == keys.size());
    for (size_t i = 0; i < keys.size(); i++) CHECK(pubs[i] == keys[i].public_key().compress());

    auto sigs = sign_compressed_batch(keys, msgs);
    CHECK(sigs.size() == keys.size());
    for (size_t i = 0; i < keys.size(); i++) {
        if (i == 4) {
            CHECK(sigs[i].status == BJJ_STATUS_MSG_RANGE);
            std::array<uint8_t, 64> zero{};
            CHECK(sigs[i].sig == zero);
            continue;
        }
        CHECK(sigs[i].status == 0);
        CHECK(sigs[i].sig == keys[i].sign(msgs[i]).compress());
    }
    bool threw = false;
    try {
        sign_compressed_batch(keys, {msgs[0]});
    } catch (const std::invalid_argument&) {
        threw = true;
    }
    CHECK(threw);
    std::printf("compressed outputs ok\n");
    return 0;
}
