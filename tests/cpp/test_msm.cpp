// msm of the C++ host mirror (host/bjj.hpp) against the reference's fold, acc.add(P_i.mul_scalar(k_i).projective()) from
// (0 : 1 : 1) then affine(), run through the mirror's own mul_scalar / add / affine; the empty sum; an off-curve point.
// Built by tests/test_msm.py; runs on the GPU box (`-m gpu`).  Exit code 0 = all passed.
#include <cstdio>
#include <string>

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
    std::vector<PrivateKey> keys(5);
    for (int k = 0; k < 5; k++)
        for (int i = 0; i < 32; i++) keys[k].key[i] = (uint8_t)(i % 10 + 31 * k);
    std::vector<Point> pts = public_batch(keys);
    pts.push_back(pts[1]);                               // a point twice
    std::vector<U256> ks;
    for (size_t i = 0; i < pts.size(); i++) {
        U256 k{};
        for (int b = 0; b < 32; b++) k[b] = (uint8_t)(0x5a ^ (b * 7 + 13 * i));
        ks.push_back(k);
    }
    ks[2] = u256_from_u64(0);
    ks[3].fill(0xff);                                    // 2^256 - 1

    PointProjective acc{u256_from_u64(0), u256_from_u64(1), u256_from_u64(1)};
    for (size_t i = 0; i < pts.size(); i++) acc = acc.add(pts[i].mul_scalar(ks[i]).projective());
    const Point want = acc.affine();
    CHECK(msm(pts, ks).equals(want));

    const Point id = msm({}, {});
    CHECK(id.equals(Point{u256_from_u64(0), u256_from_u64(1)}));

    std::vector<Point> bad = pts;
    bad[4].x[0] ^= 1;                                    // off the curve
    bool threw = false;
    try {
        msm(bad, ks);
    } catch (const Error& e) {
        threw = e.code == BJJ_ERR_ARG;
    }
    CHECK(threw);
    CHECK(msm(pts, ks).equals(want));                    // the context is clean afterwards
    std::printf("test_msm: ok\n");
    return 0;
}
