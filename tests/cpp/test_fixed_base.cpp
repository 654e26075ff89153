// FixedBase of the C++ host mirror (host/bjj.hpp) against mul_scalar_batch and the reference's addition.  Built by
// tests/test_fixed_bases.py; runs on the GPU box (`-m gpu`).  Exit code 0 = all passed.
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
    // P of the reference tests (src/lib.rs:420-459)
    Point p{from_hex_be("274dbce8d15179969bc0d49fa725bddf9de555e0ba6a693c6adb52fc9ee7a82c"),
            from_hex_be("05ce98c61b05f47fe2eae9a542bd99f6b2e78246231640b54595febfd51eb853")};
    std::vector<U256> ks;
    for (uint64_t k : {0ull, 1ull, 2ull, 3ull, 0xFFFFFFFFFFFFFFFFull}) ks.push_back(u256_from_u64(k));
    U256 top{};
    top.fill(0xFF);                                    // 2^256 - 1: the recoding's carry window
    ks.push_back(top);
    FixedBase fp(p);
    auto got = fp.mul_batch(ks);
    auto want = mul_scalar_batch(std::vector<Point>(ks.size(), p), ks);
    for (size_t i = 0; i < ks.size(); i++) CHECK(got[i].equals(want[i]));
    // k*P + l*P, and k*P + l*B8 against the reference's projective addition
    auto sum = fp.mul2_batch({u256_from_u64(2)}, &fp, {u256_from_u64(1)});
    CHECK(sum[0].equals(want[3]));
    auto b8 = fp.mul2_batch({u256_from_u64(3)}, nullptr, {u256_from_u64(5)});
    Point b8_5 = fp.mul2_batch({u256_from_u64(0)}, nullptr, {u256_from_u64(5)})[0];
    CHECK(b8[0].equals(want[3].projective().add(b8_5.projective()).affine()));
    // an off-curve point has no table
    bool threw = false;
    try {
        FixedBase bad(Point{u256_from_u64(1), u256_from_u64(1)});
    } catch (const Error& e) {
        threw = e.code == BJJ_ERR_ARG;
    }
    CHECK(threw);
    std::printf("fixed base ok\n");
    return 0;
}
