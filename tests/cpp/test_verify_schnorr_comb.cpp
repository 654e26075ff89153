// verify_schnorr_batch of the C++ host mirror (host/bjj.hpp) on sign_schnorr_batch's output as it comes: the free
// function (any key per lane), FixedBase::verify_schnorr_batch (one key) and KeySet::verify_schnorr_batch (a key per
// lane) agree with each other and with the expected outcome of every lane.  Built by tests/test_verify_schnorr_comb.py;
// runs on the GPU box (`-m gpu`).  Exit code 0 = all passed.
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
    std::vector<PrivateKey> keys(3);
    for (int k = 0; k < 3; k++)
        for (int i = 0; i < 32; i++) keys[k].key[i] = (uint8_t)(i % 10 + 17 * k);
    std::vector<Point> pks;
    for (const PrivateKey& k : keys) pks.push_back(k.public_key());
    const U256 q = from_hex_be("30644e72e131a029b85045b68181585d2833e84879b9709143e1f593f0000001");
    const std::vector<uint32_t> idx = {0, 1, 2, 1, 0, 2};
    std::vector<U256> msgs = {u256_from_u64(0x0908070605040302ull), u256_from_u64(0), q, from_hex_be("1234567890abcdef"),
                              u256_from_u64(7), u256_from_u64(99)};
    const int nonce_words = 32;                          // the reference's 1024-bit nonces: s is 40 words
    std::vector<uint32_t> nonces(nonce_words * idx.size());
    for (size_t j = 0; j < nonces.size(); j++) nonces[j] = (uint32_t)(0x9E3779B9u * (j + 1));
    std::vector<PrivateKey> signers;
    for (uint32_t j : idx) signers.push_back(keys[j]);
    auto sigs = sign_schnorr_batch(signers, msgs, nonces, nonce_words);
    for (const auto& s : sigs) CHECK(s.status == 0 && s.s.size() == 4 * 40);
    sigs[3].s[0] ^= 1;                                   // corrupted s
    msgs[4][0] ^= 1;                                     // another msg
    U256 over = q;
    over[0] += 1;
    msgs[5] = over;                                      // msg > Q: Err

    std::vector<Point> gathered;
    for (uint32_t j : idx) gathered.push_back(pks[j]);
    std::vector<uint8_t> st;
    auto ok = verify_schnorr_batch(gathered, msgs, sigs, &st);
    const std::vector<uint8_t> expect = {1, 1, 1, 0, 0, 0}, sexpect = {0, 0, 0, 0, 0, BJJ_STATUS_MSG_RANGE};
    CHECK(ok == expect);
    CHECK(st == sexpect);

    KeySet ks(pks);
    std::vector<uint8_t> kst;
    CHECK(ks.verify_schnorr_batch(idx, msgs, sigs, &kst) == expect);
    CHECK(kst == sexpect);

    FixedBase base(pks[0]);
    std::vector<SignSchnorrResult> s0 = {sigs[0], sigs[4]};
    std::vector<U256> m0 = {msgs[0], msgs[4]};
    const std::vector<uint8_t> e0 = {1, 0};
    CHECK(base.verify_schnorr_batch(m0, s0) == e0);

    int code = 0;
    try {
        ks.verify_schnorr_batch({0, 3}, {msgs[0], msgs[0]}, {sigs[0], sigs[0]});     // index 3 is outside the set
    } catch (const Error& e) {
        code = e.code;
    }
    CHECK(code == BJJ_ERR_ARG);
    std::printf("verify_schnorr comb ok\n");
    return 0;
}
