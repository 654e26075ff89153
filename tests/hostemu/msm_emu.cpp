// TEST HARNESS ONLY -- never shipped, never loaded by the product.
//
// The lane bodies of bjj_msm_batch (msm.cuh) compiled for the HOST with BJJ_HOST_EMU and driven in the order that
// launch_msm_points / msm_end (bjj_cuda.cu) launch them: prepare, a stable sort of the pairs by key (what
// cub::DeviceRadixSort yields), the accumulate levels over runs of BJJ_MSM_RUN, the segment reduction, the window sums
// and the finish.  tests/test_msm.py checks it against the oracle's fold without a GPU.
#define BJJ_HOST_EMU 1
#include <stdlib.h>
#include <string.h>
#include <algorithm>
#include <numeric>
#include <vector>
#include "../../babyjubjub-rs_b200/csrc/msm.cuh"

using namespace bjj;

namespace bjj {
void bjj_emu_need_comb_entry(const CombEntry*, int, int) {}
}  // namespace bjj

struct EmuSums {
    MsmGeom g;
    std::vector<uint8_t> buckets, seg, wsum;
    explicit EmuSums(int bits) : g(msm_geom(bits)) {
        buckets.resize((size_t)128 * g.buckets());
        seg.resize((size_t)128 * g.windows * (g.half / BJJ_MSM_SEG));
        wsum.resize((size_t)128 * g.windows);
        PointExt id;
        ext_identity(id);
        for (size_t b = 0; b < g.buckets(); b++) msm_store_ext(buckets.data(), b, id);
    }
    // msm_end: segment reduction, window sums (in index order: the group law makes the tree's order immaterial), finish
    void end(uint32_t flags, uint8_t* rx, uint8_t* ry) {
        const size_t per_window = g.half / BJJ_MSM_SEG;
        for (size_t t = 0; t < (size_t)g.windows * per_window; t++) lane_msm_segment(buckets.data(), g, t, seg.data());
        for (int w = 0; w < g.windows; w++) {
            PointExt acc, p;
            ext_identity(acc);
            for (size_t t = 0; t < per_window; t++) {
                msm_load_ext(p, seg.data(), w * per_window + t);
                msm_add_ext(acc, acc, p);
            }
            msm_store_ext(wsum.data(), w, acc);
        }
        lane_msm_finish(wsum.data(), g, flags, rx, ry);
    }
};

// launch_msm_points for one sub-batch of m points; returns the number of accumulate levels
static int emu_points(EmuSums& s, size_t m, const uint8_t* px, const uint8_t* py, const uint8_t* k, uint8_t* status, uint32_t& flags) {
    const MsmGeom& g = s.g;
    const size_t pairs = m * g.windows;
    std::vector<CombEntry> niels(m);
    std::vector<uint32_t> keys(pairs), vals(pairs);
    for (size_t i = 0; i < m; i++) lane_msm_prepare(px, py, k, i, m, g, niels.data(), keys.data(), vals.data(), status, flags);
    std::vector<size_t> order(pairs);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return keys[a] < keys[b]; });
    std::vector<uint32_t> sk(pairs), sv(pairs);
    for (size_t j = 0; j < pairs; j++) {
        sk[j] = keys[order[j]];
        sv[j] = vals[order[j]];
    }
    size_t counts[64];
    const int levels = msm_levels(pairs, counts, 64);
    std::vector<uint32_t> bkeys[2];
    std::vector<uint8_t> bpts[2];
    for (int l = 0; l < levels; l++) {
        const size_t runs = (counts[l] + BJJ_MSM_RUN - 1) / BJJ_MSM_RUN;
        std::vector<uint32_t>& ok = bkeys[l & 1];
        std::vector<uint8_t>& op = bpts[l & 1];
        ok.assign(2 * runs, 0xDEADBEEFu);
        op.assign(128 * 2 * runs, 0xA5);
        for (size_t r = 0; r < runs; r++) {
            if (l == 0)
                lane_msm_run(MsmPairs{sk.data(), sv.data(), niels.data()}, counts[0], r, g.buckets(), s.buckets.data(), ok.data(), op.data());
            else
                lane_msm_run(MsmPartials{bkeys[(l - 1) & 1].data(), bpts[(l - 1) & 1].data()}, counts[l], r, g.buckets(), s.buckets.data(),
                             ok.data(), op.data());
        }
    }
    return levels;
}

extern "C" {

// the signed digits msm_recode / msm_digit give: 256 / bits + 1 per scalar; returns that count
int emu_msm_digits(int bits, size_t n, const uint8_t* k, int32_t* d) {
    const MsmGeom g = msm_geom(bits);
    for (size_t i = 0; i < n; i++) {
        uint32_t kw[8];
        load_u256(kw, k, i);
        Recode16 rc;
        msm_recode(rc, kw, bits);
        for (int w = 0; w < g.windows; w++) d[i * g.windows + w] = msm_digit(rc, bits, w);
    }
    return g.windows;
}

// the whole call on n points, the points fed in chunks of `chunk` (0: one) into the same buckets as the host flavour
// feeds them; returns the call's flags (BJJ_FLAG_*), *levels the accumulate levels of the largest chunk
uint32_t emu_msm(int bits, size_t n, size_t chunk, const uint8_t* px, const uint8_t* py, const uint8_t* k, uint8_t* rx, uint8_t* ry,
                 uint8_t* status, int* levels) {
    EmuSums s(bits);
    uint32_t flags = 0;
    *levels = 0;
    if (chunk == 0) chunk = n ? n : 1;
    for (size_t off = 0; off < n; off += chunk) {
        const size_t m = n - off < chunk ? n - off : chunk, o = 32 * off;
        const int l = emu_points(s, m, px + o, py + o, k + o, status + off, flags);
        if (l > *levels) *levels = l;
    }
    s.end(flags, rx, ry);
    return flags;
}

// the bucket reduction alone: window 0 holds the affine points (bx, by) (canonical, 2^(bits-1) of them; bucket j
// holds digit j + 1), every other bucket the identity; writes R = W_0 = sum_j (j + 1) * B_j
void emu_msm_bucket_reduce(int bits, const uint8_t* bx, const uint8_t* by, uint8_t* rx, uint8_t* ry) {
    EmuSums s(bits);
    for (uint32_t j = 0; j < s.g.half; j++) {
        PointAff a;
        uint32_t f = 0;
        load_fr(a.x, bx, j, f);
        load_fr(a.y, by, j, f);
        PointExt e;
        ext_from_affine(e, a);
        msm_store_ext(s.buckets.data(), j, e);
    }
    s.end(0, rx, ry);
}

}  // extern "C"
