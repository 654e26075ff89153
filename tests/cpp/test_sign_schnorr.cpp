// sign_schnorr_batch of the C++ host mirror (host/bjj.hpp) against the one-lane calls it replaces: r = B8.mul_scalar(k)
// and s = k + scalar_key * Poseidon(pk.x, pk.y, r.x, r.y, msg), for nonces below 2^256 sent at nonce_words = 32 (the
// reference's 1024-bit width).  Built by tests/test_sign_schnorr.py; runs on the GPU box (`-m gpu`).  Exit code 0 = all
// passed.
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

// k + a * b as `bytes` little-endian bytes (a, b, k: 32 bytes each)
static std::vector<uint8_t> mul_add(const U256& a, const U256& b, const U256& k, size_t bytes) {
    std::vector<uint32_t> acc(bytes, 0);
    for (int i = 0; i < 32; i++)
        for (int j = 0; j < 32; j++) acc[i + j] += (uint32_t)a[i] * b[j];
    for (int i = 0; i < 32; i++) acc[i] += k[i];
    std::vector<uint8_t> out(bytes);
    uint32_t c = 0;
    for (size_t i = 0; i < bytes; i++) {
        c += acc[i];
        out[i] = (uint8_t)c;
        c >>= 8;
    }
    return out;
}

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
    std::vector<U256> msgs = {u256_from_u64(0x0908070605040302ull), u256_from_u64(0), q, u256_from_u64(1), over,
                              from_hex_be("1234567890abcdef")};
    std::vector<U256> ks = {u256_from_u64(0), u256_from_u64(1), from_hex_be("deadbeef"), from_hex_be("ffffffffffffffffffffffff"),
                            u256_from_u64(7), from_hex_be("0123456789abcdef0123456789abcdef0123456789abcdef0123456789abcdef")};
    const int words = 32;
    std::vector<uint32_t> nonces(words * keys.size(), 0);
    for (size_t i = 0; i < keys.size(); i++)
        for (int w = 0; w < 8; w++)
            for (int b = 0; b < 4; b++) nonces[words * i + w] |= (uint32_t)ks[i][4 * w + b] << (8 * b);

    auto sigs = sign_schnorr_batch(keys, msgs, nonces, words);
    CHECK(sigs.size() == keys.size());
    const Point b8{from_hex_be("0bb77a6ad63e739b4eacb2e09d6277c12ab8d8010534e0b62893f3f6bb957051"),
                   from_hex_be("25797203f7a0b24925572e1cd16bf9edfce0051fb9e133774b3c257a872d7d8b")};
    for (size_t i = 0; i < keys.size(); i++) {
        CHECK(sigs[i].s.size() == 4 * (words + 8));
        if (i == 4) {
            CHECK(sigs[i].status == BJJ_STATUS_MSG_RANGE);
            CHECK(sigs[i].r.x == U256{} && sigs[i].r.y == U256{});
            for (uint8_t v : sigs[i].s) CHECK(v == 0);
            continue;
        }
        CHECK(sigs[i].status == 0);
        CHECK(sigs[i].r.equals(b8.mul_scalar(ks[i])));
        const Point pk = keys[i].public_key();
        U256 m = msgs[i];
        if (m == q) m = U256{};                         // msg == Q hashes as 0
        const uint8_t* ins[5] = {pk.x.data(), pk.y.data(), sigs[i].r.x.data(), sigs[i].r.y.data(), m.data()};
        U256 h;
        Engine::check(bjj_poseidon_batch(default_engine().ctx(), 5, 1, ins, h.data()), "bjj_poseidon_batch");
        CHECK(sigs[i].s == mul_add(keys[i].scalar_key(), h, ks[i], 4 * (words + 8)));
    }
    bool threw = false;
    try {
        sign_schnorr_batch(keys, msgs, std::vector<uint32_t>(8), 8);
    } catch (const std::invalid_argument&) {
        threw = true;
    }
    CHECK(threw);
    std::printf("sign_schnorr ok\n");
    return 0;
}
