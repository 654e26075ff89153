// KeySet of the C++ host mirror (host/bjj.hpp): verify_batch / verify_compressed_batch against verify_batch with the
// keys gathered per lane, mul_batch against Point::mul_scalar, and the argument errors.  Built by
// tests/test_verify_keyset.py; runs on the GPU box (`-m gpu`).  Exit code 0 = all passed.
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
    // three keys: the circomlib key of the reference's test vectors (src/lib.rs:688-738) and two others
    std::vector<PrivateKey> keys(3);
    for (int k = 0; k < 3; k++)
        for (int i = 0; i < 32; i++) keys[k].key[i] = (uint8_t)(i % 10 + 17 * k);
    std::vector<Point> pks;
    for (const PrivateKey& k : keys) pks.push_back(k.public_key());
    const U256 q = from_hex_be("30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001");
    U256 over = q;
    over[0] += 1;                                       // Q + 1: verify is false
    std::vector<U256> msgs = {u256_from_u64(0x0908070605040302ull), u256_from_u64(0), u256_from_u64(1), q,
                              from_hex_be("1234567890abcdef"), u256_from_u64(7)};
    const std::vector<uint32_t> idx = {0, 1, 2, 1, 0, 2, 1};
    std::vector<Signature> sigs;
    for (size_t i = 0; i < msgs.size(); i++) sigs.push_back(keys[idx[i]].sign(msgs[i]));
    msgs.push_back(over);                               // a valid signature under a message > Q
    sigs.push_back(sigs[1]);
    sigs[4].s[0] ^= 1;                                  // corrupted S
    sigs[5].r_b8.x[0] ^= 1;                             // R8 off the curve

    KeySet ks(pks);
    CHECK(ks.size() == 3);
    auto ok = ks.verify_batch(idx, sigs, msgs);
    std::vector<Point> gathered;
    for (uint32_t j : idx) gathered.push_back(pks[j]);
    CHECK(ok == verify_batch(gathered, sigs, msgs));
    const std::vector<uint8_t> expect = {1, 1, 1, 1, 0, 0, 0};
    CHECK(ok == expect);

    std::vector<std::array<uint8_t, 64>> packed;
    for (size_t i = 0; i < 5; i++) packed.push_back(sigs[i].compress());
    std::vector<U256> cmsgs(msgs.begin(), msgs.begin() + 5);
    std::vector<uint32_t> cidx(idx.begin(), idx.begin() + 5);
    std::vector<uint8_t> st;
    auto cok = ks.verify_compressed_batch(cidx, packed, cmsgs, &st);
    const std::vector<uint8_t> cexpect = {1, 1, 1, 1, 0}, sexpect = {0, 0, 0, 0, 0};
    CHECK(cok == cexpect);
    CHECK(st == sexpect);

    const std::vector<U256> ks_scalars = {u256_from_u64(0), u256_from_u64(1), u256_from_u64(12345), from_hex_be("ff")};
    const std::vector<uint32_t> midx = {2, 0, 1, 2};
    auto got = ks.mul_batch(midx, ks_scalars);
    for (size_t i = 0; i < got.size(); i++) CHECK(got[i].equals(pks[midx[i]].mul_scalar(ks_scalars[i])));

    int code = 0;
    try {
        ks.verify_batch({0, 3}, {sigs[0], sigs[0]}, {msgs[0], msgs[0]});     // index 3 is outside the set
    } catch (const Error& e) {
        code = e.code;
    }
    CHECK(code == BJJ_ERR_ARG);
    std::vector<Point> bad = pks;
    bad[1].x[0] ^= 1;                                   // off the curve
    std::vector<uint8_t> kst;
    code = 0;
    try {
        KeySet broken(bad, default_engine(), &kst);
    } catch (const Error& e) {
        code = e.code;
    }
    CHECK(code == BJJ_ERR_ARG);
    const std::vector<uint8_t> kexpect = {BJJ_KEY_OK, BJJ_KEY_OFF_CURVE, BJJ_KEY_OK};
    CHECK(kst == kexpect);
    std::printf("keyset ok\n");
    return 0;
}
