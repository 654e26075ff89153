// FixedBase::verify_batch / verify_compressed_batch of the C++ host mirror (host/bjj.hpp) against verify_batch with the
// key in every lane.  Built by tests/test_verify_base.py; runs on the GPU box (`-m gpu`).  Exit code 0 = all passed.
#include <cstdio>
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
    // the circomlib key of the reference's test vectors (src/lib.rs:688-738) signs every message
    PrivateKey key;
    for (int i = 0; i < 32; i++) key.key[i] = (uint8_t)(i % 10);
    const Point pk = key.public_key();
    const U256 q = from_hex_be("30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001");
    U256 over = q;
    over[0] += 1;                                       // Q + 1: verify is false
    std::vector<U256> msgs = {u256_from_u64(0x0908070605040302ull), u256_from_u64(0), u256_from_u64(1), q,
                              from_hex_be("1234567890abcdef"), u256_from_u64(7)};
    std::vector<Signature> sigs;
    for (const U256& m : msgs) sigs.push_back(key.sign(m));
    msgs.push_back(over);                               // a valid signature under a message > Q
    sigs.push_back(sigs[0]);
    sigs[4].s[0] ^= 1;                                  // corrupted S
    sigs[5].r_b8.x[0] ^= 1;                             // R8 off the curve

    FixedBase fb(pk);
    auto ok = fb.verify_batch(sigs, msgs);
    auto want = verify_batch(std::vector<Point>(sigs.size(), pk), sigs, msgs);
    CHECK(ok == want);
    const std::vector<uint8_t> expect = {1, 1, 1, 1, 0, 0, 0};
    CHECK(ok == expect);

    std::vector<std::array<uint8_t, 64>> packed;
    for (size_t i = 0; i < 5; i++) packed.push_back(sigs[i].compress());
    packed.push_back(packed[0]);
    packed.back()[31] |= 0x7F;                          // y >= Q: "y outside the Finite Field over R"
    packed.back()[30] = 0xFF;
    std::vector<U256> cmsgs(msgs.begin(), msgs.begin() + 5);
    cmsgs.push_back(msgs[0]);
    std::vector<uint8_t> st;
    auto cok = fb.verify_compressed_batch(packed, cmsgs, &st);
    const std::vector<uint8_t> cexpect = {1, 1, 1, 1, 0, 0}, sexpect = {0, 0, 0, 0, 0, BJJ_STATUS_Y_RANGE};
    CHECK(cok == cexpect);
    CHECK(st == sexpect);
    bool threw = false;
    try {
        fb.verify_batch(sigs, {msgs[0]});
    } catch (const std::invalid_argument&) {
        threw = true;
    }
    CHECK(threw);
    std::printf("verify base ok\n");
    return 0;
}
