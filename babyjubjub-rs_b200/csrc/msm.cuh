// Lane bodies of the multi-scalar product R = sum_i k_i * P_i (bjj_msm_batch, kernels in k_msm.cu).
//
// Bucket method (Pippenger) with signed c-bit windows, c = 8 or 16 (msm_window_bits picks it from n):
//   1. prepare: every point is checked (canonical, on the curve), converted to the affine Niels form of the a = -1 model
//      (96 B, a CombEntry) and its scalar recoded into WINDOWS signed digits (recode8 / recode16, the last window the
//      recoding carry).  Each (point, window) emits one pair: key = the bucket w * HALF + |d| - 1, value = the point's
//      index with the digit's sign in bit 31.  A zero digit, and every digit of an off-curve point, gets the discard key
//      WINDOWS * HALF, so the pair count (and with it every launch) depends on n only.
//   2. the pairs are sorted by key (cub::DeviceRadixSort over the key's bits).
//   3. accumulate: the sorted list is cut into runs of BJJ_MSM_RUN pairs, one thread per run.  A bucket that begins and
//      ends inside a run is added into the bucket array directly; the partial sums of the first and the last bucket of
//      a run that continue into the neighbouring runs go to a boundary list (two slots per run), which is itself sorted
//      by key and is reduced by the same pass, level after level, until it fits one run.  Every thread adds at most
//      BJJ_MSM_RUN points, however the digits are distributed: with every scalar equal, one bucket per window holds all
//      n points and its sum still spreads over n / BJJ_MSM_RUN threads.
//   4. bucket reduce: W_w = sum_b b * B_{w,b} by running sums over segments of BJJ_MSM_SEG buckets, then a tree per window.
//   5. finish: R = sum_w 2^(c w) W_w by Horner's rule, one inversion, canonical (x, y) on the original curve.
// Every point on the curve has an order dividing ORDER, so the raw 256-bit k_i is exact, and the group law of the a = -1
// model is complete: any grouping of the sum gives the reference's fold (include/bjj_cuda.h, bjj_msm_batch).
#pragma once
#include "lanes.cuh"

namespace bjj {

#define BJJ_FLAG_OFF_CURVE 4u        // a point of bjj_msm_batch is off the curve (bjj_sync: BJJ_ERR_ARG)
#define BJJ_MSM_RUN 32               // sorted pairs per accumulate thread
#define BJJ_MSM_SEG 32               // buckets per running-sum segment of the bucket reduction
#define BJJ_MSM_DUMMY 0x80000000u    // boundary-list key bit: the slot holds no partial sum
#define BJJ_MSM_NEG 0x80000000u      // pair value bit: subtract the point

// window geometry: c bits, WINDOWS = 256 / c + 1 (the last holds the recoding carry), HALF = 2^(c-1) buckets per window
struct MsmGeom {
    int bits, windows;
    uint32_t half;
    BJJ_HD uint32_t buckets() const { return (uint32_t)windows * half; }      // also the discard key
};
BJJ_HD MsmGeom msm_geom(int bits) {
    MsmGeom g;
    g.bits = bits;
    g.windows = 256 / bits + 1;
    g.half = 1u << (bits - 1);
    return g;
}

// the signed digits of k: d[w] in [-HALF, HALF) for w < WINDOWS - 1, d[WINDOWS - 1] in {0, 1}
BJJ_HD int msm_digit(const Recode16& rc, int bits, int w) {
    const int last = 256 / bits;
    if (w == last) return (int)rc.top;
    return bits == 16 ? recode16_digit(rc, w) : recode8_digit(*reinterpret_cast<const Recode8*>(&rc), w);
}
BJJ_HD void msm_recode(Recode16& rc, const uint32_t* k, int bits) {
    if (bits == 16)
        recode16(rc, k);
    else
        recode8(*reinterpret_cast<Recode8*>(&rc), k);
}

// pair key of digit d in window w (the discard key for d = 0)
BJJ_HD uint32_t msm_key(const MsmGeom& g, int w, int d) {
    if (d == 0) return g.buckets();
    return (uint32_t)w * g.half + (uint32_t)(d < 0 ? -d : d) - 1;
}

// point i of a sub-batch of m points: status byte (BJJ_KEY_*), flags, its Niels entry and its WINDOWS pairs at
// keys[w * m + i], vals[w * m + i]
BJJ_HD void lane_msm_prepare(const uint8_t* px, const uint8_t* py, const uint8_t* k, size_t i, size_t m, const MsmGeom& g,
                             CombEntry* niels, uint32_t* keys, uint32_t* vals, uint8_t* status, uint32_t& flags) {
    PointAff p;
    uint32_t f = 0;
    load_fr(p.x, px, i, f);
    load_fr(p.y, py, i, f);
    const bool on = on_curve(p);
    status[i] = f ? 2 : on ? 0 : 1;     // BJJ_KEY_NONCANONICAL outranks BJJ_KEY_OFF_CURVE, as in bjj_keyset_create
    if (!on) f |= BJJ_FLAG_OFF_CURVE;
    flags |= f;
    PointExt e;
    ext_from_affine(e, p);
    comb_store_niels(niels + i, e.X, e.Y);
    uint32_t kw[8];
    load_u256(kw, k, i);
    Recode16 rc;
    msm_recode(rc, kw, g.bits);
#pragma unroll 1
    for (int w = 0; w < g.windows; w++) {
        const int d = on ? msm_digit(rc, g.bits, w) : 0;
        keys[(size_t)w * m + i] = msm_key(g, w, d);
        vals[(size_t)w * m + i] = (uint32_t)i | (d < 0 ? BJJ_MSM_NEG : 0u);
    }
}

// extended points in memory: 4 x 32 B raw Montgomery limbs (X, Y, Z, T) per point
BJJ_HD void msm_load_ext(PointExt& p, const uint8_t* base, size_t i) {
    load_u256(p.X.v, base, 4 * i);
    load_u256(p.Y.v, base, 4 * i + 1);
    load_u256(p.Z.v, base, 4 * i + 2);
    load_u256(p.T.v, base, 4 * i + 3);
}
BJJ_HD void msm_store_ext(uint8_t* base, size_t i, const PointExt& p) {
    store_u256(base, 4 * i, p.X.v);
    store_u256(base, 4 * i + 1, p.Y.v);
    store_u256(base, 4 * i + 2, p.Z.v);
    store_u256(base, 4 * i + 3, p.T.v);
}
// r = a + b for two extended points (9M)
BJJ_HD void msm_add_ext(PointExt& r, const PointExt& a, const PointExt& b) {
    Niels n;
    niels_from_ext(n, b);
    ext_add_niels<true>(r, a, n);
}

// the input of one accumulate level: the sorted pairs (level 1: a Niels entry per pair, signed) or the boundary list of
// the level before (an extended point per slot)
struct MsmPairs {
    const uint32_t* keys;
    const uint32_t* vals;
    const CombEntry* niels;
    BJJ_HD bool dummy(size_t j, uint32_t nb) const { return keys[j] >= nb; }
    BJJ_HD void add(PointExt& acc, size_t j) const {
        const uint32_t v = vals[j];
        NielsAff n;
        comb_fetch<Comb8>(n, niels, 0, (int)(v & ~BJJ_MSM_NEG));
        niels_aff_cneg(n, (v & BJJ_MSM_NEG) != 0);
        ext_add_niels_aff<true>(acc, acc, n);
    }
};
struct MsmPartials {
    const uint32_t* keys;
    const uint8_t* pts;
    BJJ_HD bool dummy(size_t j, uint32_t nb) const { return (keys[j] & BJJ_MSM_DUMMY) || keys[j] >= nb; }
    BJJ_HD void add(PointExt& acc, size_t j) const {
        PointExt p;
        msm_load_ext(p, pts, j);
        msm_add_ext(acc, acc, p);
    }
};

// run r of a level with `count` entries: the entries [r * RUN, min((r + 1) * RUN, count)).  Writes its closed buckets
// into `buckets` (adding to what they hold: the chunks of one call share the buckets) and its two boundary slots
// out_keys / out_pts[2r], [2r + 1]: the partial of a bucket open to the left in the first, of one open to the right in
// the second (a run that is one bucket open on either side uses the first), else the slot's bucket key | DUMMY.
template <class In>
BJJ_HD void lane_msm_run(const In& in, size_t count, size_t r, uint32_t nb, uint8_t* buckets, uint32_t* out_keys, uint8_t* out_pts) {
    const size_t s = r * BJJ_MSM_RUN, e = s + BJJ_MSM_RUN < count ? s + BJJ_MSM_RUN : count;
    const uint32_t kmask = ~BJJ_MSM_DUMMY;
    const uint32_t first_key = in.keys[s] & kmask, last_key = in.keys[e - 1] & kmask;
    const bool open_left = s > 0 && (in.keys[s - 1] & kmask) == first_key;
    const bool open_right = e < count && (in.keys[e] & kmask) == last_key;
    out_keys[2 * r] = first_key | BJJ_MSM_DUMMY;
    out_keys[2 * r + 1] = last_key | BJJ_MSM_DUMMY;
    PointExt acc;
    ext_identity(acc);
    bool real = false, first = true;
    uint32_t cur = first_key;
#pragma unroll 1
    for (size_t j = s;; j++) {
        const bool end = j == e;
        const uint32_t key = end ? 0 : in.keys[j] & kmask;
        if (end || key != cur) {
            // close the segment of bucket `cur`: 0 = into the bucket, 1 / 2 = boundary slot 2r / 2r + 1
            const int where = first ? ((open_left || (end && open_right)) ? 1 : 0) : (end && open_right) ? 2 : 0;
            if (real) {
                if (where == 0) {
                    PointExt b;
                    msm_load_ext(b, buckets, cur);
                    msm_add_ext(b, b, acc);
                    msm_store_ext(buckets, cur, b);
                } else {
                    out_keys[2 * r + where - 1] = cur;
                    msm_store_ext(out_pts, 2 * r + where - 1, acc);
                }
            }
            if (end) break;
            first = false;
            real = false;
            ext_identity(acc);
            cur = key;
        }
        if (!in.dummy(j, nb)) {
            in.add(acc, j);
            real = true;
        }
    }
}

// the entry counts of the accumulate levels of a sub-batch with `pairs` pairs: level 1 reads the pairs, level l + 1 the
// 2 * ceil(count_l / RUN) boundary slots of level l; the last level fits one run.  Returns the number of levels.
BJJ_HD int msm_levels(size_t pairs, size_t* counts, int max_levels) {
    int l = 0;
    size_t c = pairs;
    for (;;) {
        if (l < max_levels) counts[l] = c;
        l++;
        if (c <= BJJ_MSM_RUN) return l;
        c = 2 * ((c + BJJ_MSM_RUN - 1) / BJJ_MSM_RUN);
    }
}

// segment t of the bucket reduction: buckets j0 .. j0 + SEG - 1 of window w (bucket j holds digit j + 1) ->
// sum_j (j + 1) * B_j, by the running sums acc = sum_j (j + 1 - j0) * B_j, S = sum_j B_j and acc + j0 * S
BJJ_HD void lane_msm_segment(const uint8_t* buckets, const MsmGeom& g, size_t t, uint8_t* seg_out) {
    const uint32_t per_window = g.half / BJJ_MSM_SEG;
    const uint32_t w = (uint32_t)(t / per_window), j0 = (uint32_t)(t % per_window) * BJJ_MSM_SEG;
    PointExt run, acc, b;
    ext_identity(run);
    ext_identity(acc);
#pragma unroll 1
    for (int j = BJJ_MSM_SEG - 1; j >= 0; j--) {
        msm_load_ext(b, buckets, (size_t)w * g.half + j0 + j);
        msm_add_ext(run, run, b);
        msm_add_ext(acc, acc, run);
    }
    // j0 * S, MSB first (j0 < 2^15)
    PointExt m;
    ext_identity(m);
    Niels ns;
    niels_from_ext(ns, run);
#pragma unroll 1
    for (int bit = 15; bit >= 0; bit--) {
        ext_dbl<true>(m, m);
        if ((j0 >> bit) & 1) ext_add_niels<true>(m, m, ns);
    }
    msm_add_ext(acc, acc, m);
    msm_store_ext(seg_out, t, acc);
}

// R = sum_w 2^(c w) W_w (Horner), written as canonical affine (x, y) on the original curve, or (0, 0) when a point was
// off the curve
BJJ_HD void lane_msm_finish(const uint8_t* wsum, const MsmGeom& g, uint32_t flags, uint8_t* rx, uint8_t* ry) {
    PointExt acc, p;
    msm_load_ext(acc, wsum, g.windows - 1);
#pragma unroll 1
    for (int w = g.windows - 2; w >= 0; w--) {
#pragma unroll 1
        for (int i = 0; i < g.bits; i++) ext_dbl<true>(acc, acc);
        msm_load_ext(p, wsum, w);
        msm_add_ext(acc, acc, p);
    }
    if (flags & BJJ_FLAG_OFF_CURVE) {
        uint32_t z[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        store_u256(rx, 0, z);
        store_u256(ry, 0, z);
        return;
    }
    store_ext_affine(rx, ry, 0, acc);
}

}  // namespace bjj
