// Per-lane bodies of the batch kernels.  One lane = one element of the SoA batch.
//
// Boundary layout (include/bjj_cuda.h): every field element / scalar / compressed point is 32 bytes
// little-endian at byte offset 32*i of its own array (SoA), i.e. 8 x u32 = two 16-byte vector loads
// per lane, 1 KiB contiguous per warp.
//
// Each lane function cites the reference item it replaces (paths into /root/reference).
#pragma once
#include <string.h>
#include "blake512.cuh"
#include "curve.cuh"
#include "fr.cuh"
#include "poseidon.cuh"
#include "split.cuh"

namespace bjj {

struct alignas(16) U128 {
    uint32_t x, y, z, w;
};

// ---- lane I/O -------------------------------------------------------------------------------------
BJJ_HD void load_u256(uint32_t* w, const uint8_t* base, size_t i) {
#if BJJ_DEVICE_CODE
    const uint4* p = reinterpret_cast<const uint4*>(base + 32 * i);
    uint4 a = __ldg(p), b = __ldg(p + 1);
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
    w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
#else
    memcpy(w, base + 32 * i, 32);
#endif
}
BJJ_HD void store_u256(uint8_t* base, size_t i, const uint32_t* w) {
#if BJJ_DEVICE_CODE
    uint4* p = reinterpret_cast<uint4*>(base + 32 * i);
    p[0] = make_uint4(w[0], w[1], w[2], w[3]);
    p[1] = make_uint4(w[4], w[5], w[6], w[7]);
#else
    memcpy(base + 32 * i, w, 32);
#endif
}

// status / error bits -------------------------------------------------------------------------------
// per-lane status byte of decompress (maps 1:1 to the reference's error strings)
#define BJJ_ST_OK 0
#define BJJ_ST_Y_RANGE 1      // "y outside the Finite Field over R"   src/lib.rs:202
#define BJJ_ST_NO_INV 2       // "no mod inv of Zero"                  src/utils.rs:14
#define BJJ_ST_NOT_SQUARE 3   // "not a mod p square"                  src/utils.rs:119
#define BJJ_ST_MSG_RANGE 4    // "msg outside the Finite Field"        src/lib.rs:310, :366
// batch-level flag bits (device word OR-ed by lanes)
#define BJJ_FLAG_NONCANONICAL 1u   // a field-element input was >= Q (cannot happen through the Rust types)

// canonical bytes -> Montgomery; *flags |= NONCANONICAL if the integer is >= Q (value is reduced)
BJJ_HD void load_fr(Fr& r, const uint8_t* base, size_t i, uint32_t& flags) {
    Fr raw;
    load_u256(raw.v, base, i);
    const uint32_t q[8] = BJJ_LIMBS8(BJJ_Q);
    if (!u256_lt(raw.v, q)) flags |= BJJ_FLAG_NONCANONICAL;
    fr_to_mont(r, raw);
}
BJJ_HD void store_fr(uint8_t* base, size_t i, const Fr& a) {
    Fr c;
    fr_from_mont(c, a);
    store_u256(base, i, c.v);
}

// ---- per-thread window table in global memory --------------------------------------------------------
// 9 Niels entries (0 = identity, j = j*P) x 8 x 16 B, interleaved across threads:
//   U128 index = (entry*8 + q) * stride + slot       (q = coordinate*2 + half)
struct LaneTable {
    U128* base;
    size_t stride;
    size_t slot;
};
#define BJJ_TABLE_ENTRIES 9
#define BJJ_TABLE_U128_PER_LANE (BJJ_TABLE_ENTRIES * 8)

BJJ_HD void table_store(const LaneTable& t, int e, const Niels& n) {
    const Fr* f[4] = {&n.ypx, &n.ymx, &n.t2d, &n.z2};
#pragma unroll
    for (int c = 0; c < 4; c++) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
            U128 u;
            u.x = f[c]->v[4 * h + 0];
            u.y = f[c]->v[4 * h + 1];
            u.z = f[c]->v[4 * h + 2];
            u.w = f[c]->v[4 * h + 3];
            t.base[(size_t)(e * 8 + c * 2 + h) * t.stride + t.slot] = u;
        }
    }
}
BJJ_HD void table_load(Niels& n, const LaneTable& t, int e) {
    Fr* f[4] = {&n.ypx, &n.ymx, &n.t2d, &n.z2};
#pragma unroll
    for (int c = 0; c < 4; c++) {
#pragma unroll
        for (int h = 0; h < 2; h++) {
            U128 u = t.base[(size_t)(e * 8 + c * 2 + h) * t.stride + t.slot];
            f[c]->v[4 * h + 0] = u.x;
            f[c]->v[4 * h + 1] = u.y;
            f[c]->v[4 * h + 2] = u.z;
            f[c]->v[4 * h + 3] = u.w;
        }
    }
}

// entries 0..8 = j*P
BJJ_HD void table_build(const LaneTable& t, const PointExt& p) {
    Niels n, n1;
    niels_identity(n);
    table_store(t, 0, n);
    niels_from_ext(n1, p);
    table_store(t, 1, n1);
    PointExt acc = p;      // 2P is P + P by the (complete) addition: same cost as a doubling, no second formula
#pragma unroll 1
    for (int j = 2; j <= 8; j++) {
        ext_add_niels<true>(acc, acc, n1);
        niels_from_ext(n, acc);
        table_store(t, j, n);
    }
}

// signed digit d in [-8, 8] -> Niels of d*P
BJJ_HD void table_select(Niels& n, const LaneTable& t, int d) {
    int ad = d < 0 ? -d : d;
    table_load(n, t, ad);
    niels_cneg(n, d < 0);
}

// ---- fixed-base comb for B8 (and for caller points, bjj_base_create) ------------------------------------
// comb[w][j] = j * 65536^w * B8 as affine Niels (y+x, y-x, 2d'xy) on the a = -1 model, j = 0..32768,
// w = 0..16 (w = 16 only holds j = 0, 1 for the recoding carry): 16 x 32,769 x 96 B = 50 MB, L2-resident,
// gathered with ld.global.nc.  Built once per context on the device (k_comb_build, ~15 ms); a caller point's table
// is the same with B8 replaced by that point (k_comb_build_point).  Signed 16-bit
// digits make a fixed-base multiplication 17 mixed additions and no doubling; verify adds its B8 term (w * B8, the
// one full-width scalar left after the split) the same way, after the Straus pass over the two per-lane points.
#define BJJ_COMB_BITS 16
#define BJJ_COMB_WINDOWS 17
#define BJJ_COMB_ENTRIES 32769
#define BJJ_COMB_TOTAL ((size_t)(BJJ_COMB_WINDOWS - 1) * BJJ_COMB_ENTRIES + 2)
#if !BJJ_DEVICE_CODE && defined(BJJ_HOST_EMU)
// the host test harness fills table entries on demand instead of building all 524,290 of them
void bjj_emu_need_comb_entry(const struct CombEntry* comb, int w, int j);
#endif
struct CombEntry {   // 96 bytes
    uint32_t ypx[8], ymx[8], t2d[8];
};

// the raw entry |d| of window w (no sign applied yet)
BJJ_HD void comb_fetch(NielsAff& n, const CombEntry* comb, int w, int d) {
    int ad = d < 0 ? -d : d;
    const CombEntry* e = comb + (size_t)w * BJJ_COMB_ENTRIES + ad;
#if !BJJ_DEVICE_CODE && defined(BJJ_HOST_EMU)
    bjj_emu_need_comb_entry(comb, w, ad);
#endif
#if BJJ_DEVICE_CODE
    const uint4* p = reinterpret_cast<const uint4*>(e);
    uint4 q0 = __ldg(p), q1 = __ldg(p + 1), q2 = __ldg(p + 2), q3 = __ldg(p + 3), q4 = __ldg(p + 4), q5 = __ldg(p + 5);
    n.ypx.v[0] = q0.x; n.ypx.v[1] = q0.y; n.ypx.v[2] = q0.z; n.ypx.v[3] = q0.w;
    n.ypx.v[4] = q1.x; n.ypx.v[5] = q1.y; n.ypx.v[6] = q1.z; n.ypx.v[7] = q1.w;
    n.ymx.v[0] = q2.x; n.ymx.v[1] = q2.y; n.ymx.v[2] = q2.z; n.ymx.v[3] = q2.w;
    n.ymx.v[4] = q3.x; n.ymx.v[5] = q3.y; n.ymx.v[6] = q3.z; n.ymx.v[7] = q3.w;
    n.t2d.v[0] = q4.x; n.t2d.v[1] = q4.y; n.t2d.v[2] = q4.z; n.t2d.v[3] = q4.w;
    n.t2d.v[4] = q5.x; n.t2d.v[5] = q5.y; n.t2d.v[6] = q5.z; n.t2d.v[7] = q5.w;
#else
    fr_set(n.ypx, e->ypx);
    fr_set(n.ymx, e->ymx);
    fr_set(n.t2d, e->t2d);
#endif
}
BJJ_HD void comb_select(NielsAff& n, const CombEntry* comb, int w, int d) {
    comb_fetch(n, comb, w, d);
    niels_aff_cneg(n, d < 0);
}

// acc += k * base (comb = the table of base) for a 256-bit k: 17 mixed additions, no doublings.  `from_identity` starts
// acc at the identity, after the recoding as fixed_base_comb always did (so its kernels compile as before);
// lane_fixed_base2 runs two walks over two tables into one accumulator.  BJJ_COMB_PREFETCH: the entry of window w - 1
// is requested before the addition of window w, so that its L2 latency (the 50 MB table is gathered at random) runs
// under ~900 multiplier instructions instead of in front of them.
#ifndef BJJ_COMB_PREFETCH
#define BJJ_COMB_PREFETCH 1
#endif
BJJ_HD void fixed_base_comb_acc(PointExt& acc, const CombEntry* comb, const uint32_t* k, bool from_identity = false) {
    Recode16 rc;
    recode16(rc, k);
    if (from_identity) ext_identity(acc);
#if BJJ_COMB_PREFETCH
    NielsAff cur, nxt;
    int d = (int)rc.top;
    comb_fetch(cur, comb, BJJ_COMB_WINDOWS - 1, d);
#pragma unroll 1
    for (int w = BJJ_COMB_WINDOWS - 2; w >= 0; w--) {
        const int dn = recode16_digit(rc, w);
        comb_fetch(nxt, comb, w, dn);
        niels_aff_cneg(cur, d < 0);
        ext_add_niels_aff<true>(acc, acc, cur);
        cur = nxt;
        d = dn;
    }
    niels_aff_cneg(cur, d < 0);
    ext_add_niels_aff<true>(acc, acc, cur);
#else
    NielsAff n;
    comb_select(n, comb, BJJ_COMB_WINDOWS - 1, (int)rc.top);
    ext_add_niels_aff<true>(acc, acc, n);
#pragma unroll 1
    for (int w = BJJ_COMB_WINDOWS - 2; w >= 0; w--) {
        comb_select(n, comb, w, recode16_digit(rc, w));
        ext_add_niels_aff<true>(acc, acc, n);
    }
#endif
}
BJJ_HD void fixed_base_comb(PointExt& acc, const CombEntry* comb, const uint32_t* k) {
    fixed_base_comb_acc(acc, comb, k, true);
}

// one comb entry: j * 65536^w * p for an on-curve p of the original curve   (one thread per (w, j)).  Every on-curve
// point has an order dividing ORDER < 2^254, so the table serves every 256-bit scalar like B8's does.
BJJ_HD void comb_build_entry(CombEntry* comb, int w, int j, const PointAff& p) {
    CombEntry* e = comb + (size_t)w * BJJ_COMB_ENTRIES + j;
    PointExt base, acc;
    ext_from_affine(base, p);
#pragma unroll 1
    for (int i = 0; i < BJJ_COMB_BITS * w; i++) ext_dbl<true>(base, base);
    ext_identity(acc);
    Niels nb;
    niels_from_ext(nb, base);
#pragma unroll 1
    for (int bit = BJJ_COMB_BITS - 1; bit >= 0; bit--) {
        ext_dbl<true>(acc, acc);
        if ((j >> bit) & 1) ext_add_niels<true>(acc, acc, nb);
    }
    // affine on the a = -1 model, then Niels form
    Fr zi, x, y, t;
    fr_inv(zi, acc.Z);
    fr_mul(x, acc.X, zi);
    fr_mul(y, acc.Y, zi);
    fr_mul(t, x, y);
    const Fr d2 = fr_const(BJJ_TWO_DP_M);
    fr_mul(t, t, d2);
    Fr ypx, ymx;
    fr_add(ypx, y, x);
    fr_sub(ymx, y, x);
    fr_reduce(ypx);
    fr_reduce(ymx);
    fr_reduce(t);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        e->ypx[i] = ypx.v[i];
        e->ymx[i] = ymx.v[i];
        e->t2d[i] = t.v[i];
    }
}
// the context's B8 table (k_comb_build)
BJJ_HD void comb_build_entry(CombEntry* comb, int w, int j) {
    PointAff b8;
    b8.x = fr_const(BJJ_B8X_M);
    b8.y = fr_const(BJJ_B8Y_M);
    comb_build_entry(comb, w, j, b8);
}

// outcome of building a caller point's table (k_comb_build_point)
#define BJJ_BASE_OK 0
#define BJJ_BASE_OFF_CURVE 1
#define BJJ_BASE_NONCANONICAL 2

// ---- affine output ------------------------------------------------------------------------------------
// a = -1 extended -> canonical affine bytes on the original curve (Fermat inverse per lane)
BJJ_HD void store_ext_affine(uint8_t* rx, uint8_t* ry, size_t i, const PointExt& p) {
    PointProj pj;
    ext_to_proj(pj, p);
    PointAff a;
    proj_affine(a, pj);
    store_fr(rx, i, a.x);
    store_fr(ry, i, a.y);
}

// Batched affine conversion (replaces one Fr::inverse per point, src/lib.rs:78, by Montgomery's trick):
// the point kernels park (X/sqrt(-a) : Y : Z) in scratch as raw Montgomery limbs; a second kernel gives
// every thread the lanes t, t+T, t+2T, .. and spends ONE Fermat inversion per thread:
//   forward:  p_i = p_(i-T) * z_i (stored);   inv = 1 / p_last;
//   backward: 1/z_i = inv * p_(i-T);  inv *= z_i;   x_i = X_i / z_i,  y_i = Y_i / z_i.
// Z == 0 keeps the reference rule of PointProjective::affine (src/lib.rs:71-76): the lane yields (0, 0)
// and is left out of the product.  Off-curve lanes of mul_scalar park Z = 0 and are overwritten by the
// exact-lane kernel afterwards.
struct ProjScratch {
    uint8_t* x;
    uint8_t* y;
    uint8_t* z;
    uint8_t* p;    // running products
};

BJJ_HD void store_ext_scratch(const ProjScratch& s, size_t i, const PointExt& p) {
    PointProj pj;
    ext_to_proj(pj, p);
    store_u256(s.x, i, pj.x.v);
    store_u256(s.y, i, pj.y.v);
    store_u256(s.z, i, pj.z.v);
}
BJJ_HD void store_zero_scratch(const ProjScratch& s, size_t i) {
    Fr z;
    fr_zero(z);
    store_u256(s.x, i, z.v);
    store_u256(s.y, i, z.v);
    store_u256(s.z, i, z.v);
}

// (A warp-cooperative variant of the inversion below -- prefix/suffix products across the 32 lanes by shuffles, one
// Fermat inversion of the warp's total -- was measured and dropped: under SIMT the 32 per-thread inversions of a warp
// already ARE one instruction stream, so sharing it buys nothing and the 12 extra multiplications cost: public_batch
// 341 -> 322 M keys/s.  What amortises the inversion is lanes per thread.  Two independent product chains per thread,
// merged before the one inversion, were measured as well: 2.570 against 2.564 ms per 2^20 keys at 32 lanes per thread,
// 2.61 / 2.88 ms at 64 / 128 lanes per thread -- the kernel lives on the number of resident warps, and lanes per thread
// take them away.  profiles/r2_ab_exact_early_chunks.txt.)
//
// `Out` is the output form, fixed at compile time: out(i, x, y) receives lane i's affine (x, y) in Montgomery form
// ((0, 0) for Z == 0).  AffineOut stores the two coordinates, CompressedOut stores Point::compress of them.
template <class Out>
BJJ_HD void batch_affine_strided(const ProjScratch& s, Out out, size_t n, size_t t, size_t T) {
    const Fr one = fr_const(BJJ_ONE_M);
    Fr acc = one, z;
    size_t last = t;
    if (t >= n) return;
#pragma unroll 1
    for (size_t i = t; i < n; i += T) {
        load_u256(z.v, s.z, i);
        if (!fr_is_zero(z)) fr_mul(acc, acc, z);
        store_u256(s.p, i, acc.v);
        last = i;
    }
    Fr inv;
    fr_inv(inv, acc);
#pragma unroll 1
    for (size_t i = last;; i -= T) {
        Fr prev = one, zi, x, y;
        if (i >= t + T) load_u256(prev.v, s.p, i - T);
        load_u256(z.v, s.z, i);
        const bool zero = fr_is_zero(z);
        fr_mul(zi, inv, prev);
        if (!zero) fr_mul(inv, inv, z);
        load_u256(x.v, s.x, i);
        load_u256(y.v, s.y, i);
        fr_mul(x, x, zi);
        fr_mul(y, y, zi);
        if (zero) {
            fr_zero(x);
            fr_zero(y);
        }
        out(i, x, y);
        if (i < t + T) break;
    }
}

// Point::compress's sign rule (src/lib.rs:166-178): bit 255 of the compressed y is set when x > Q/2 (x, y canonical)
BJJ_HD void compress_sign(uint32_t* y, const uint32_t* x) {
    if (u256_lt(BJJ_QHALF, x)) y[7] |= 0x80000000u;
}

struct AffineOut {
    uint8_t *rx, *ry;
    BJJ_HD void operator()(size_t i, const Fr& x, const Fr& y) const {
        store_fr(rx, i, x);
        store_fr(ry, i, y);
    }
};
struct CompressedOut {
    uint8_t* out32;
    BJJ_HD void operator()(size_t i, const Fr& x, const Fr& y) const {
        Fr cx, cy;
        fr_from_mont(cx, x);
        fr_from_mont(cy, y);
        compress_sign(cy.v, cx.v);
        store_u256(out32, i, cy.v);
    }
};

BJJ_HD void batch_affine_strided(const ProjScratch& s, uint8_t* rx, uint8_t* ry, size_t n, size_t t, size_t T) {
    batch_affine_strided(s, AffineOut{rx, ry}, n, t, T);
}

// ---- lane bodies --------------------------------------------------------------------------------------

// test hook for Fr (reference Fr ops: mul_assign / square / add_assign / sub_assign / inverse)
#define BJJ_FR_OP_MUL 0
#define BJJ_FR_OP_ADD 1
#define BJJ_FR_OP_SUB 2
#define BJJ_FR_OP_INV 3
#define BJJ_FR_OP_SQR 4
#define BJJ_FR_OP_SQR_LAZY 5
BJJ_HD void lane_fr_op(int op, const uint8_t* a, const uint8_t* b, uint8_t* out, size_t i, uint32_t& flags) {
    Fr x, y, r;
    load_fr(x, a, i, flags);
    load_fr(y, b, i, flags);
    switch (op) {
        case BJJ_FR_OP_MUL: fr_mul(r, x, y); break;
        case BJJ_FR_OP_ADD: fr_add(r, x, y); break;
        case BJJ_FR_OP_SUB: fr_sub(r, x, y); break;
        case BJJ_FR_OP_INV: fr_inv(r, x); break;
        case BJJ_FR_OP_SQR_LAZY: {      // the squaring on the upper half of the lazy domain: (x mod Q) + Q in [Q, 2Q)
            const uint32_t q[8] = BJJ_LIMBS8(BJJ_Q);
            fr_reduce(x);
            add256(x.v, x.v, q);
            fr_sqr(r, x);
            break;
        }
        default: fr_sqr(r, x); break;
    }
    store_fr(out, i, r);
}

// PointProjective::add (src/lib.rs:88-131), projective in, projective out, literal formula
BJJ_HD void lane_add(const uint8_t* px, const uint8_t* py, const uint8_t* pz, const uint8_t* qx,
                     const uint8_t* qy, const uint8_t* qz, uint8_t* rx, uint8_t* ry, uint8_t* rz, size_t i,
                     uint32_t& flags) {
    PointProj p, q, r;
    load_fr(p.x, px, i, flags);
    load_fr(p.y, py, i, flags);
    load_fr(p.z, pz, i, flags);
    load_fr(q.x, qx, i, flags);
    load_fr(q.y, qy, i, flags);
    load_fr(q.z, qz, i, flags);
    proj_add_bbjlp(r, p, q);
    store_fr(rx, i, r.x);
    store_fr(ry, i, r.y);
    store_fr(rz, i, r.z);
}

// PointProjective::affine (src/lib.rs:70-85)
BJJ_HD void lane_affine(const uint8_t* px, const uint8_t* py, const uint8_t* pz, uint8_t* rx, uint8_t* ry,
                        size_t i, uint32_t& flags) {
    PointProj p;
    load_fr(p.x, px, i, flags);
    load_fr(p.y, py, i, flags);
    load_fr(p.z, pz, i, flags);
    PointAff a;
    proj_affine(a, p);
    store_fr(rx, i, a.x);
    store_fr(ry, i, a.y);
}

// windowed variable-base ladder on the a = -1 model: acc = n * p  (p on the curve, n any 256-bit integer)
BJJ_HD void var_base_mul(PointExt& acc, const PointExt& p, const uint32_t* n, const LaneTable& tbl) {
    table_build(tbl, p);
    Recode4 rc;
    recode4(rc, n);
    Niels nn;
    ext_identity(acc);
    table_select(nn, tbl, (int)rc.top);
    ext_add_niels<false>(acc, acc, nn);
#pragma unroll 1
    for (int i = 63; i >= 0; i--) {
        ext_dbl<false>(acc, acc);
        ext_dbl<false>(acc, acc);
        ext_dbl<false>(acc, acc);
        ext_dbl<true>(acc, acc);
        table_select(nn, tbl, recode4_digit(rc, i));
        ext_add_niels<false>(acc, acc, nn);
    }
}

BJJ_HD int clz32(uint32_t x) {
#if BJJ_DEVICE_CODE
    return __clz((int)x);
#else
    return __builtin_clz(x);
#endif
}

// exact lane: the reference sequence, bit for bit (off-curve inputs).  Point::mul_scalar,
// src/lib.rs:149-164: r = (0,1,1); exp = P; for bit i of n, LSB first, up to bits(n): if set
// r = r.add(exp); exp = exp.add(exp);  then r.affine().
BJJ_HD_NOINLINE void mul_scalar_exact(PointAff& r, const PointAff& p, const uint32_t* n, int nwords) {
    PointProj acc, e;
    fr_zero(acc.x);
    acc.y = fr_const(BJJ_ONE_M);
    acc.z = fr_const(BJJ_ONE_M);
    e.x = p.x;
    e.y = p.y;
    e.z = fr_const(BJJ_ONE_M);
    int nb = 0;     // BigInt::bits()
    for (int i = 0; i < nwords; i++)
        if (n[i]) nb = 32 * i + (32 - clz32(n[i]));
    // The exact lanes are few and latency-bound (fewer than two such warps per SMSP), and in a warp the lanes'
    // bits differ anyway: r + exp is computed every step next to exp + exp -- two independent dependency
    // chains in one basic block -- and kept only where the bit is set.
#pragma unroll 1
    for (int i = 0; i < nb; i++) {
        const bool bit = (n[i >> 5] >> (i & 31)) & 1;
        PointProj t, e2;
        proj_add_bbjlp(t, acc, e);
        proj_add_bbjlp(e2, e, e);
        fr_cmov(acc.x, t.x, bit);
        fr_cmov(acc.y, t.y, bit);
        fr_cmov(acc.z, t.z, bit);
        e = e2;
    }
    proj_affine(r, acc);
}

// Queue of lanes that failed the on-curve gate.  The fast kernel only records their indices; a second,
// small kernel replays the reference sequence for them, so the fast kernel carries neither the exact
// path's registers nor its divergence.
struct ExactQueue {
    uint32_t* count;
    uint32_t* list;
};
BJJ_HD void exact_push(const ExactQueue& q, size_t i) {
#if BJJ_DEVICE_CODE
    uint32_t slot = atomicAdd(q.count, 1u);
#else
    uint32_t slot = (*q.count)++;
#endif
    q.list[slot] = (uint32_t)i;
}

// Point::mul_scalar (src/lib.rs:149-164): on-curve gate -> fast ladder, else queued for the exact lane.
BJJ_HD void lane_mul_scalar(const uint8_t* px, const uint8_t* py, const uint8_t* scalar, const ProjScratch& scr,
                            size_t i, const LaneTable& tbl, const ExactQueue& q, uint32_t& flags) {
    PointAff p;
    load_fr(p.x, px, i, flags);
    load_fr(p.y, py, i, flags);
    if (!on_curve(p)) {
        store_zero_scratch(scr, i);      // Z = 0: skipped by the batched affine pass, written by the exact kernel
        exact_push(q, i);
        return;
    }
    uint32_t n[8];
    load_u256(n, scalar, i);
    PointExt e, acc;
    ext_from_affine(e, p);
    var_base_mul(acc, e, n, tbl);
    store_ext_scratch(scr, i, acc);
}

// Scalars wider than 256 bits (the reference's n is a BigInt of any size): element i of a wide array is `nwords`
// 32-bit little-endian words, nwords a multiple of 8 up to BJJ_MAX_SCALAR_WORDS.
#define BJJ_MAX_SCALAR_WORDS 64

// out = x mod ORDER for a wide x: on-curve points have order dividing ORDER = 8 * SUBORDER, so the fast ladder may use
// the reduced scalar (exact).  Shift-and-subtract, MSB first; ORDER < 2^254, so 2 * acc + 1 fits 256 bits.
BJJ_HD void lane_reduce_scalar_order(const uint8_t* wide, int nwords, uint8_t* out32, size_t i) {
    uint32_t acc[8], t[8];
#pragma unroll
    for (int k = 0; k < 8; k++) acc[k] = 0;
#pragma unroll 1
    for (int blk = (nwords >> 3) - 1; blk >= 0; blk--) {
        uint32_t w[8];
        load_u256(w, wide, i * (size_t)(nwords >> 3) + (size_t)blk);
#pragma unroll 1
        for (int bit = 255; bit >= 0; bit--) {
            uint32_t b = 0;
#pragma unroll
            for (int j = 0; j < 8; j++) b = ((bit >> 5) == j) ? w[j] : b;
            b = (b >> (bit & 31)) & 1u;
#pragma unroll
            for (int k = 7; k > 0; k--) acc[k] = (acc[k] << 1) | (acc[k - 1] >> 31);
            acc[0] = (acc[0] << 1) | b;
            const uint32_t borrow = sub256(t, acc, BJJ_ORDER);
#pragma unroll
            for (int k = 0; k < 8; k++) acc[k] = borrow ? acc[k] : t[k];
        }
    }
    store_u256(out32, i, acc);
}

// exact lane of mul_scalar: lane index taken from the queue; the scalar is read at its full width
BJJ_HD void lane_mul_scalar_exact(const uint8_t* px, const uint8_t* py, const uint8_t* scalar, int nwords, uint8_t* rx,
                                  uint8_t* ry, size_t i) {
    uint32_t flags = 0;
    PointAff p, r;
    load_fr(p.x, px, i, flags);
    load_fr(p.y, py, i, flags);
    uint32_t n[BJJ_MAX_SCALAR_WORDS];
#pragma unroll 1
    for (int b = 0; b < (nwords >> 3); b++) load_u256(n + 8 * b, scalar, i * (size_t)(nwords >> 3) + (size_t)b);
    mul_scalar_exact(r, p, n, nwords);
    store_fr(rx, i, r.x);
    store_fr(ry, i, r.y);
}

// B8.mul_scalar(k) for a raw 256-bit scalar (src/lib.rs:305, :329, :405)
BJJ_HD void lane_fixed_base(const uint8_t* scalar, const ProjScratch& scr, size_t i, const CombEntry* comb) {
    uint32_t k[8];
    load_u256(k, scalar, i);
    PointExt acc;
    fixed_base_comb(acc, comb, k);
    store_ext_scratch(scr, i, acc);
}

// (k * P).projective().add((l * Q).projective()).affine() (src/lib.rs:70-131, 149-164) for on-curve P, Q with tables
// comb_p, comb_q: both products are group elements and the reference's addition is complete on the curve, so the
// result is the group sum, accumulated in one point (34 mixed additions)
BJJ_HD void lane_fixed_base2(const uint8_t* k, const uint8_t* l, const ProjScratch& scr, size_t i, const CombEntry* comb_p,
                             const CombEntry* comb_q) {
    uint32_t s[8];
    PointExt acc;
    ext_identity(acc);
    load_u256(s, k, i);
    fixed_base_comb_acc(acc, comb_p, s);
    load_u256(s, l, i);
    fixed_base_comb_acc(acc, comb_q, s);
    store_ext_scratch(scr, i, acc);
}

// entry (w, j) of the table of the caller point (px, py) (bytes of element 0): every thread checks the point, builds
// its entry only for a valid one, and returns the BJJ_BASE_* outcome
BJJ_HD uint32_t lane_comb_build_point(CombEntry* comb, int w, int j, const uint8_t* px, const uint8_t* py) {
    PointAff p;
    uint32_t flags = 0;
    load_fr(p.x, px, 0, flags);
    load_fr(p.y, py, 0, flags);
    const uint32_t st = flags ? BJJ_BASE_NONCANONICAL : on_curve(p) ? BJJ_BASE_OK : BJJ_BASE_OFF_CURVE;
    if (st == BJJ_BASE_OK) comb_build_entry(comb, w, j, p);
    return st;
}

// PrivateKey::public (src/lib.rs:304-306) = B8 * scalar_key(key)
BJJ_HD void lane_public(const uint8_t* key, const ProjScratch& scr, size_t i, const CombEntry* comb) {
    uint32_t kw[8], k[8];
    load_u256(kw, key, i);
    scalar_key_from_key(k, kw);
    PointExt acc;
    fixed_base_comb(acc, comb, k);
    store_ext_scratch(scr, i, acc);
}

// PrivateKey::scalar_key (src/lib.rs:284-302) test hook
BJJ_HD void lane_scalar_key(const uint8_t* key, uint8_t* out, size_t i) {
    uint32_t kw[8], k[8];
    load_u256(kw, key, i);
    scalar_key_from_key(k, kw);
    store_u256(out, i, k);
}

// Point::compress (src/lib.rs:166-178)
BJJ_HD void lane_compress(const uint8_t* px, const uint8_t* py, uint8_t* out, size_t i, uint32_t& flags) {
    uint32_t x[8], y[8];
    load_u256(x, px, i);
    load_u256(y, py, i);
    const uint32_t q[8] = BJJ_LIMBS8(BJJ_Q);
    if (!u256_lt(x, q) || !u256_lt(y, q)) flags |= BJJ_FLAG_NONCANONICAL;
    compress_sign(y, x);
    store_u256(out, i, y);
}

// a^((T-1)/2) driven by the public exponent bits
BJJ_HD uint32_t ph_lookup(const Fr& t) {
    Fr c = t;
    fr_reduce(c);
    return BJJ_PH_LUT[(c.v[0] * BJJ_PH_HASH_MULT) >> 23];
}

// decompress_point (src/lib.rs:192-224) with utils::modinv / modsqrt (src/utils.rs:11-29, 109-160).
// The reference's Tonelli-Shanks loop is replaced by a fixed schedule: x0 = a^((T+1)/2), b = a^T lies in
// the order-2^28 subgroup; its discrete log k is found 7 bits at a time (Pohlig-Hellman with table
// look-ups) and x = x0 * g^(-k/2).  The returned x does not depend on which root a sqrt algorithm finds
// (src/lib.rs:217-220 fixes the sign), so the result is bit-identical.
// The decompression is split around the one modular inverse so that a batch can share it
// (Montgomery's trick, lanes.cuh::batch_inverse_strided):
//   decompress_prepare: range check, u = 1 - y^2, v = a - d y^2           -> status, y, u, v
//   decompress_finish : x^2 = u / v, fixed-schedule square root, sign rule -> status, x
BJJ_HD uint32_t decompress_prepare(Fr& ym, Fr& u, Fr& v, const uint32_t* bytes) {
    uint32_t yw[8];
#pragma unroll
    for (int i = 0; i < 8; i++) yw[i] = bytes[i];
    yw[7] &= 0x7FFFFFFFu;
    const uint32_t q[8] = BJJ_LIMBS8(BJJ_Q);
    if (!u256_lt(yw, q)) return BJJ_ST_Y_RANGE;
    Fr yraw;
    fr_set(yraw, yw);
    fr_to_mont(ym, yraw);
    const Fr one = fr_const(BJJ_ONE_M), cA = fr_const(BJJ_A_M), cD = fr_const(BJJ_D_M);
    Fr y2;
    fr_sqr(y2, ym);
    fr_sub(u, one, y2);
    fr_mul(v, cD, y2);
    fr_sub(v, cA, v);
    if (fr_is_zero(v)) return BJJ_ST_NO_INV;
    return BJJ_ST_OK;
}

BJJ_HD uint32_t decompress_finish(Fr& xm, bool sign, const Fr& u, const Fr& vinv) {
    Fr a;
    fr_mul(a, u, vinv);
    if (fr_is_zero(a)) return BJJ_ST_NOT_SQUARE;     // modsqrt rejects a == 0 (src/utils.rs:118)
    Fr w, x0, b, t;
#if BJJ_POW_SCHED
    fr_pow_sched(w, a, BJJ_POW_TM1H, BJJ_POW_TM1H_STEPS, BJJ_POW_TM1H_TAIL);
#else
    fr_pow(w, a, BJJ_EXP_TM1H, BJJ_EXP_TM1H_BITS);
#endif
    fr_mul(x0, a, w);
    fr_mul(b, x0, w);
    uint32_t k[4];
#pragma unroll 1
    for (int j = 0; j < 4; j++) {
        t = b;
#pragma unroll 1
        for (int s = 0; s < 21 - 7 * j; s++) fr_sqr(t, t);
        k[j] = ph_lookup(t);
        if (k[j] > 127) return BJJ_ST_NOT_SQUARE;
        if (j == 0 && (k[0] & 1)) return BJJ_ST_NOT_SQUARE;    // odd discrete log: non-residue
        Fr c = fr_const(BJJ_PH_NEG[j][k[j]]);
        fr_mul(b, b, c);
        Fr hc = fr_const(BJJ_PH_HALF[j][k[j]]);
        fr_mul(x0, x0, hc);
    }
    fr_sqr(t, x0);
    if (!fr_eq(t, a)) return BJJ_ST_NOT_SQUARE;
    // sign rule (src/lib.rs:217-220): negate iff (x > Q>>1) != sign
    Fr xc;
    fr_from_mont(xc, x0);
    const bool big = u256_lt(BJJ_QHALF, xc.v);
    if (big != sign) fr_neg(x0, x0);
    xm = x0;
    return BJJ_ST_OK;
}

// single-lane composition (exact lanes, tests): one Fermat inverse
BJJ_HD uint32_t decompress_core(Fr& xm, Fr& ym, const uint32_t* bytes) {
    Fr u, v, vi;
    uint32_t st = decompress_prepare(ym, u, v, bytes);
    if (st != BJJ_ST_OK) return st;
    fr_inv(vi, v);
    return decompress_finish(xm, (bytes[7] >> 31) != 0, u, vi);
}

// Batched form.  Compressed point of lane i = 32-byte element i * stride + off of `in` (1, 0 for a plain
// array; 2, 0 for the R8 half of sig64).  Phase 1 parks u, v (v = 0 for rejected lanes) and the early
// status (one byte per slot in the scratch's y area) in scratch.
BJJ_HD void lane_decompress_prepare(const uint8_t* in, size_t stride, size_t off, const ProjScratch& scr, size_t slot,
                                    size_t i) {
    uint32_t b[8];
    load_u256(b, in, i * stride + off);
    Fr y, u, v;
    fr_zero(u);
    fr_zero(v);
    uint32_t st = decompress_prepare(y, u, v, b);
    if (st != BJJ_ST_OK) fr_zero(v);
    store_u256(scr.x, slot, u.v);
    store_u256(scr.z, slot, v.v);
    scr.y[slot] = (uint8_t)st;
}

// in-place inversion of scr.z[t], scr.z[t+T], ... (zeros stay zero); one Fermat inversion per thread
BJJ_HD void batch_inverse_strided(const ProjScratch& s, size_t n, size_t t, size_t T) {
    const Fr one = fr_const(BJJ_ONE_M);
    Fr acc = one, z;
    size_t last = t;
    if (t >= n) return;
#pragma unroll 1
    for (size_t i = t; i < n; i += T) {
        load_u256(z.v, s.z, i);
        if (!fr_is_zero(z)) fr_mul(acc, acc, z);
        store_u256(s.p, i, acc.v);
        last = i;
    }
    Fr inv;
    fr_inv(inv, acc);
#pragma unroll 1
    for (size_t i = last;; i -= T) {
        Fr prev = one, zi;
        if (i >= t + T) load_u256(prev.v, s.p, i - T);
        load_u256(z.v, s.z, i);
        if (!fr_is_zero(z)) {
            fr_mul(zi, inv, prev);
            fr_mul(inv, inv, z);
            store_u256(s.z, i, zi.v);
        }
        if (i < t + T) break;
    }
}

// Phase 3: x from (u, 1/v).  `merge` (second point of verify_compressed): an earlier error of the same
// lane (R8 is decoded first) wins, as in decompress_signature followed by decompress_point.
BJJ_HD void lane_decompress_finish(const uint8_t* in, size_t stride, size_t off, const ProjScratch& scr, size_t slot,
                                   uint8_t* rx, uint8_t* ry, uint8_t* status, size_t i, bool merge) {
    uint32_t own = scr.y[slot];
    Fr x, y;
    fr_zero(x);
    fr_zero(y);
    if (own == BJJ_ST_OK) {
        uint32_t b[8];
        load_u256(b, in, i * stride + off);
        const bool sign = (b[7] >> 31) != 0;
        b[7] &= 0x7FFFFFFFu;
        Fr yraw, u, vi;
        fr_set(yraw, b);
        fr_to_mont(y, yraw);
        load_u256(u.v, scr.x, slot);
        load_u256(vi.v, scr.z, slot);
        own = decompress_finish(x, sign, u, vi);
        if (own != BJJ_ST_OK) {
            fr_zero(x);
            fr_zero(y);
        }
    }
    store_fr(rx, i, x);
    store_fr(ry, i, y);
    if (!merge)
        status[i] = (uint8_t)own;
    else if (status[i] == BJJ_ST_OK)
        status[i] = (uint8_t)own;
}

BJJ_HD void lane_decompress(const uint8_t* in, uint8_t* rx, uint8_t* ry, uint8_t* status, size_t i) {
    uint32_t b[8];
    load_u256(b, in, i);
    Fr x, y;
    fr_zero(x);
    fr_zero(y);
    uint32_t st = decompress_core(x, y, b);
    if (st != BJJ_ST_OK) {
        fr_zero(x);
        fr_zero(y);
    }
    store_fr(rx, i, x);
    store_fr(ry, i, y);
    status[i] = (uint8_t)st;
}

// POSEIDON.hash(inputs) for NIN = T-1 inputs (src/lib.rs:400-401 uses NIN = 5)
template <int T>
BJJ_HD void lane_poseidon(const uint8_t* const* in, uint8_t* out, size_t i, uint32_t& flags) {
    Fr st[T];
    fr_zero(st[0]);
#pragma unroll
    for (int j = 1; j < T; j++) load_fr(st[j], in[j - 1], i, flags);
    poseidon_permute<T>(st);
    store_fr(out, i, st[0]);
}

// x (nwords <= 24 32-bit limbs) mod SUBORDER, canonical.  x = x0 + x1 R + x2 R^2 with R = 2^256: each part is brought
// below 2l by one Montgomery product with R, R^2, R^3 mod l (split.cuh::montmul_suborder: a * b / R mod l), the sum is
// below 6l < 2^254 and three conditional subtractions (4l, 2l, l) finish.  (The signer reduces the 512-bit nonce hash
// and the 576-bit r + hm * 8 sk; a bit-serial shift-and-subtract here cost 14 % of a signature.)
BJJ_HD void mod_suborder(uint32_t* out, const uint32_t* x, int nwords) {
    uint32_t part[8], acc[8], t[8];
#pragma unroll
    for (int i = 0; i < 8; i++) acc[i] = 0;
#pragma unroll 1
    for (int p = 0; p < 3; p++) {
        if (8 * p >= nwords) break;
#pragma unroll
        for (int i = 0; i < 8; i++) part[i] = (8 * p + i < nwords) ? x[8 * p + i] : 0u;
        montmul_suborder(t, part, p == 0 ? BJJ_L_R1 : (p == 1 ? BJJ_L_R2 : BJJ_L_R3));
        add256(acc, acc, t);
    }
#pragma unroll 1
    for (int k = 2; k >= 0; k--) {          // acc -= (l << k) where that keeps it non-negative
        uint32_t lk[8];
        u256_shl(lk, BJJ_SUBORDER, k);
        uint32_t borrow = sub256(t, acc, lk);
#pragma unroll
        for (int i = 0; i < 8; i++) acc[i] = borrow ? acc[i] : t[i];
    }
#pragma unroll
    for (int i = 0; i < 8; i++) out[i] = acc[i];
}

// PrivateKey::sign (src/lib.rs:308-342).  status: 0 ok, 4 = "msg outside the Finite Field" (:310).
//   h = BLAKE512(key); r = BLAKE512(h[32..64] || msg_le32) mod SUBORDER; R8 = B8*r; A = public();
//   hm = Poseidon(R8.x, R8.y, A.x, A.y, msg);  S = (r + hm * (scalar_key << 3)) mod SUBORDER
// the two scalars of a signature: sk = scalar_key(key), r = BLAKE512(h[32..64] || msg_le32) mod SUBORDER
BJJ_HD void sign_scalars(uint32_t* sk, uint32_t* r, const uint32_t* key, const uint32_t* msg) {
    uint64_t le[4], h[8], m2[8], h2[8];
#pragma unroll
    for (int i = 0; i < 4; i++) le[i] = (uint64_t)key[2 * i] | ((uint64_t)key[2 * i + 1] << 32);
    blake512_short<4>(h, le);
    scalar_key_from_digest(sk, h);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        m2[i] = h[4 + i];                                                        // digest bytes 32..63
        m2[4 + i] = bswap64((uint64_t)msg[2 * i] | ((uint64_t)msg[2 * i + 1] << 32));   // msg, 32 LE bytes
    }
    blake512_short_be<8>(h2, m2);
    uint32_t rw[16];
#pragma unroll
    for (int i = 0; i < 8; i++) {          // the 64 digest bytes read as a little-endian integer
        uint64_t l = bswap64(h2[i]);
        rw[2 * i] = (uint32_t)l;
        rw[2 * i + 1] = (uint32_t)(l >> 32);
    }
    mod_suborder(r, rw, 16);
}

// S = (r + hm * (sk << 3)) mod SUBORDER, hm the canonical integer of the hash
BJJ_HD void sign_finish(uint32_t* s_out, const uint32_t* hm, const uint32_t* sk, const uint32_t* r) {
    // prod = hm * (sk << 3) + r   (8 x 9 limbs -> 17 limbs)
    uint32_t sk8[9], prod[18];
    sk8[0] = sk[0] << 3;
#pragma unroll
    for (int i = 1; i < 8; i++) sk8[i] = (sk[i] << 3) | (sk[i - 1] >> 29);
    sk8[8] = sk[7] >> 29;
#pragma unroll
    for (int i = 0; i < 18; i++) prod[i] = 0;
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
        uint64_t c = 0;
#pragma unroll 1
        for (int j = 0; j < 9; j++) {
            c += (uint64_t)hm[i] * sk8[j] + prod[i + j];
            prod[i + j] = (uint32_t)c;
            c >>= 32;
        }
        prod[i + 9] = (uint32_t)c;
    }
    uint64_t c = 0;
#pragma unroll 1
    for (int i = 0; i < 18; i++) {
        c += (uint64_t)prod[i] + (i < 8 ? r[i] : 0u);
        prod[i] = (uint32_t)c;
        c >>= 32;
    }
    mod_suborder(s_out, prod, 18);
}

// One lane start to finish (the host test harness and the fused k_sign; the library's bjj_sign_batch runs the same
// steps as a pipeline of kernels, see bjj_cuda.cu::launch_sign).
BJJ_HD uint32_t sign_core(PointExt& r8, uint32_t* s_out, const uint32_t* key, const uint32_t* msg,
                          const CombEntry* comb, Fr& r8x_m, Fr& r8y_m) {
    const uint32_t q[8] = BJJ_LIMBS8(BJJ_Q);
    if (u256_lt(q, msg)) return BJJ_ST_MSG_RANGE;
    uint32_t sk[8], r[8];
    sign_scalars(sk, r, key, msg);
    fixed_base_comb(r8, comb, r);
    PointExt a;
    fixed_base_comb(a, comb, sk);
    // affine coordinates of R8 and A on the original curve: both Z are non-zero (complete formulas on curve points),
    // so ONE inversion of Z_R * Z_A serves both
    PointProj pr, pa;
    PointAff r8a, aa;
    ext_to_proj(pr, r8);
    ext_to_proj(pa, a);
    {
        Fr t, ti, zr, za;
        fr_mul(t, pr.z, pa.z);
        fr_inv(ti, t);
        fr_mul(zr, ti, pa.z);
        fr_mul(za, ti, pr.z);
        fr_mul(r8a.x, pr.x, zr);
        fr_mul(r8a.y, pr.y, zr);
        fr_mul(aa.x, pa.x, za);
        fr_mul(aa.y, pa.y, za);
    }
    Fr st[6], mraw;
    fr_zero(st[0]);
    st[1] = r8a.x;
    st[2] = r8a.y;
    st[3] = aa.x;
    st[4] = aa.y;
    fr_set(mraw, msg);
    fr_to_mont(st[5], mraw);
    poseidon_permute<6>(st);
    Fr hm;
    fr_from_mont(hm, st[0]);
    sign_finish(s_out, hm.v, sk, r);
    r8x_m = r8a.x;
    r8y_m = r8a.y;
    return BJJ_ST_OK;
}

// ---- the same signature as a pipeline (bjj_cuda.cu::launch_sign) -----------------------------------------------
// phase 1: status, the two scalars, and a copy of msg that is 0 where msg is out of range (so that the Poseidon kernel
// neither hashes nor flags it)
BJJ_HD void lane_sign_scalars(const uint8_t* key32, const uint8_t* msg32, uint8_t* sk_out, uint8_t* r_out, uint8_t* msg_out,
                              uint8_t* status, size_t i) {
    uint32_t key[8], msg[8], sk[8], r[8];
    load_u256(key, key32, i);
    load_u256(msg, msg32, i);
    const uint32_t q[8] = BJJ_LIMBS8(BJJ_Q);
    const bool bad = u256_lt(q, msg), eq_q = u256_eq(q, msg);
    sign_scalars(sk, r, key, msg);
#pragma unroll
    for (int k = 0; k < 8; k++) {
        sk[k] = bad ? 0u : sk[k];
        r[k] = bad ? 0u : r[k];
        msg[k] = (bad || eq_q) ? 0u : msg[k];        // msg == Q is accepted and hashes as 0 (Fr::from_str reduces it)
    }
    store_u256(sk_out, i, sk);
    store_u256(r_out, i, r);
    store_u256(msg_out, i, msg);
    status[i] = bad ? (uint8_t)BJJ_ST_MSG_RANGE : (uint8_t)BJJ_ST_OK;
}
// last phase: S from the hash; rejected lanes return zeros like the fused lane.  `Out` is the output form, fixed at
// compile time: out.reject(i, zero) for a lane whose status is not OK, out.accept(i, S) otherwise.
template <class Out>
BJJ_HD void lane_sign_finish(const uint8_t* hm32, const uint8_t* sk32, const uint8_t* r32, const uint8_t* status, Out out,
                             size_t i) {
    uint32_t hm[8], sk[8], r[8], s[8];
    if (status[i] != BJJ_ST_OK) {
#pragma unroll
        for (int k = 0; k < 8; k++) s[k] = 0;
        out.reject(i, s);
        return;
    }
    load_u256(hm, hm32, i);
    load_u256(sk, sk32, i);
    load_u256(r, r32, i);
    sign_finish(s, hm, sk, r);
    out.accept(i, s);
}
// R8 is already in r8x, r8y (the fixed-base pass wrote it there); S goes to s32
struct SignOut {
    uint8_t *r8x, *r8y, *s32;
    BJJ_HD void reject(size_t i, const uint32_t* zero) const {
        store_u256(r8x, i, zero);
        store_u256(r8y, i, zero);
        store_u256(s32, i, zero);
    }
    BJJ_HD void accept(size_t i, const uint32_t* s) const { store_u256(s32, i, s); }
};
// Signature::compress (src/lib.rs:245-257): compress(R8) || S into lane i of the 64-byte-stride sig64; R8 is read from
// the canonical affine planes r8x, r8y
struct SignCompressedOut {
    const uint8_t *r8x, *r8y;
    uint8_t* sig64;
    BJJ_HD void reject(size_t i, const uint32_t* zero) const {
        store_u256(sig64, 2 * i, zero);
        store_u256(sig64, 2 * i + 1, zero);
    }
    BJJ_HD void accept(size_t i, const uint32_t* s) const {
        uint32_t x[8], y[8];
        load_u256(x, r8x, i);
        load_u256(y, r8y, i);
        compress_sign(y, x);
        store_u256(sig64, 2 * i, y);
        store_u256(sig64, 2 * i + 1, s);
    }
};
BJJ_HD void lane_sign_finish(const uint8_t* hm32, const uint8_t* sk32, const uint8_t* r32, const uint8_t* status, uint8_t* r8x,
                             uint8_t* r8y, uint8_t* s32, size_t i) {
    lane_sign_finish(hm32, sk32, r32, status, SignOut{r8x, r8y, s32}, i);
}

BJJ_HD void lane_sign(const uint8_t* key32, const uint8_t* msg32, uint8_t* r8x, uint8_t* r8y, uint8_t* s32,
                      uint8_t* status, size_t i, const CombEntry* comb) {
    uint32_t key[8], msg[8], s[8];
    load_u256(key, key32, i);
    load_u256(msg, msg32, i);
    PointExt r8;
    Fr x, y;
    fr_zero(x);
    fr_zero(y);
#pragma unroll
    for (int k = 0; k < 8; k++) s[k] = 0;
    uint32_t st = sign_core(r8, s, key, msg, comb, x, y);
    store_fr(r8x, i, x);
    store_fr(r8y, i, y);
    store_u256(s32, i, s);
    status[i] = (uint8_t)st;
}

// verify (src/lib.rs:395-412).  Returns 0/1 like the reference's bool.
//   msg > Q -> false; hm = Poseidon(R8.x, R8.y, A.x, A.y, msg mod Q);
//   accept iff  S*B8 == R8 + (8*hm)*A   compared in affine coordinates.
// Fast lane (A and R8 on the curve): the group equation  S*B8 - R8 - hm*(8A) == O  multiplied by an odd v with
//   u = v*hm, w = v*S (mod l) half-size (split.cuh): one Straus pass over  u*(-+8A) + |v|*(-R8),  then  + w*B8  from the
//   comb, and the test is  sum == O = (0 : 1 : 1)  checked projectively (no inversion).
// Exact lane (any input point off the curve): the reference sequence replayed literally, in a second
// kernel fed by the ExactQueue.
// mode selects the signature scheme sharing this pipeline:
//   BJJ_MODE_EDDSA   verify          (src/lib.rs:395-412): hm = H(R8.x, R8.y, A.x, A.y, msg),  S*B8 == R8 + (8*hm)*A
//   BJJ_MODE_SCHNORR verify_schnorr  (src/lib.rs:364-385): h  = H(pk.x, pk.y, r.x, r.y, msg),  s*B8 == r + h*pk
// (`a` is the public key and `r8` the commitment point in both).
#define BJJ_MODE_EDDSA 0
#define BJJ_MODE_SCHNORR 1
#define BJJ_MODE_NEVER 0x5a5a5a5a   // no caller passes it: guards the pipe-selection ballast of vm.cuh
BJJ_HD void verify_hm(Fr& hm, const PointAff& r8, const PointAff& a, const Fr& msg_m, int mode) {
    Fr st[6];
    fr_zero(st[0]);
    const bool sch = mode == BJJ_MODE_SCHNORR;
    st[1] = r8.x;
    st[2] = r8.y;
    st[3] = a.x;
    st[4] = a.y;
    fr_cmov(st[1], a.x, sch);
    fr_cmov(st[2], a.y, sch);
    fr_cmov(st[3], r8.x, sch);
    fr_cmov(st[4], r8.y, sch);
    st[5] = msg_m;
    poseidon_permute<6>(st);
    fr_from_mont(hm, st[0]);      // canonical integer hm < Q
}

// Scalars of one pending lane, written by the hash kernel (see split.cuh):
//   u = v * hm (mod l) >= 0,  |v| odd with its sign in bit 255 of the stored word,  w = |v| * S (mod l).
// verify_schnorr lanes (and BJJ_VERIFY_SPLIT=0) carry u = hm, v = 1, w = S.
struct VerifyScalars {
    uint32_t u[8], v[8], w[8];
    uint32_t vneg;
};

// number of radix-16 windows a recoded scalar occupies (index of its highest non-zero digit + 1; 65 = carry)
BJJ_HD int recode4_windows(const Recode4& rc) {
    int n = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) {
        const uint32_t x = rc.w[k] ^ 0x88888888u;
        if (x) n = 8 * k + ((35 - BJJ_CLZ32(x)) >> 2);
    }
    return rc.top ? 65 : n;
}
BJJ_HD int recode4_digit_any(const Recode4& rc, int i) {   // i in [0, 64]
    return i == 64 ? (int)rc.top : recode4_digit(rc, i);
}

// requires A and R8 ON the curve.  Accepts iff  w*B8 - |v|*R8 - sign(v)*u*(8A) == O  (EdDSA; Schnorr: pk for 8A),
// which for the scalars above is the reference's  S*B8 == R8 + (8*hm)*A.
// One Straus pass over the two per-lane points (radix-16 tables in global memory) runs as many windows as
// the wider of u, |v| needs (32-33 after the split, 64-65 without); w * B8 is 17 additions from the
// fixed-base table afterwards.
// Recoded scalars parked outside the register file (shared memory on the device): word k of scalar s sits at
// base[(9 * s + k) * stride]; word 8 is the recoding carry.  27 registers less for the Straus loop to carry.
struct ScalarPark {
    uint32_t* base;
    int stride;
};
#define BJJ_PARK_WORDS 27
BJJ_HD void park_store(const ScalarPark& pk, int s, const uint32_t* w, uint32_t top) {
#pragma unroll
    for (int k = 0; k < 8; k++) pk.base[(9 * s + k) * pk.stride] = w[k];
    pk.base[(9 * s + 8) * pk.stride] = top;
}
BJJ_HD int park_digit4(const ScalarPark& pk, int s, int i) {      // signed radix-16 digit i in [0, 64]
    const uint32_t w = pk.base[(9 * s + (i >> 3)) * pk.stride];
    return i == 64 ? (int)w : (int)((w >> ((i & 7) * 4)) & 15u) - 8;
}
BJJ_HD int park_digit16(const ScalarPark& pk, int s, int i) {     // signed radix-65536 digit i in [0, 16]
    const uint32_t w = pk.base[(9 * s + (i >> 1)) * pk.stride];
    return i == 16 ? (int)w : (int)((w >> ((i & 1) * 16)) & 65535u) - 32768;
}

BJJ_HD uint32_t verify_fast(const PointAff& r8, const PointAff& a, const VerifyScalars& sc, const LaneTable& tbl_a,
                            const LaneTable& tbl_r, const CombEntry* comb, int mode, const ScalarPark& park) {
    PointExt acc;
    // tables of -sign(v) * 8A (pk itself for Schnorr, which multiplies pk by h) and of -R8.  Every loop below is
    // kept rolled: the kernel holds one inlined copy of the doubling and one of the addition (see curve.cuh).
#pragma unroll 1
    for (int t = 0; t < 2; t++) {
        PointExt p;
        ext_from_affine(p, t == 0 ? a : r8);
        if (t == 0 && mode == BJJ_MODE_EDDSA) {
#pragma unroll 1
            for (int j = 0; j < 3; j++) ext_dbl_rt(p, p, j == 2);
        }
        if (t == 1 || !sc.vneg) {       // negate: (-X, Y, Z, -T)
            fr_neg(p.X, p.X);
            fr_neg(p.T, p.T);
        }
        LaneTable tb = tbl_a;
        if (t == 1) tb.base = tbl_r.base;
        table_build(tb, p);
    }
    int nwin;
    {
        Recode4 ru, rv;
        recode4(ru, sc.u);
        recode4(rv, sc.v);
        Recode16 rw;
        recode16(rw, sc.w);
        nwin = recode4_windows(ru);
        const int nv = recode4_windows(rv);
        nwin = nwin > nv ? nwin : nv;
        park_store(park, 0, ru.w, ru.top);
        park_store(park, 1, rv.w, rv.top);
        park_store(park, 2, rw.w, rw.top);
    }
    // Uniform trip counts matter beyond divergence: the warps of an SM share the instruction cache only while
    // they run the same stretch of the (large) loop body below, and a warp that finishes a lane one window early
    // is out of step for good -- with per-warp counts of 32-34 this kernel ran 2x slower (no_instruction stalls
    // 2.0 per issue against 0.85).  33 windows cover all but ~0.2 % of the split scalars.
    nwin = nwin < 33 ? 33 : nwin;
#if BJJ_DEVICE_CODE
    // one trip count per warp: the lanes stay converged and reach the B8 windows together (the extra leading
    // digits of a narrower lane are zero = the identity entry)
    nwin = __reduce_max_sync(__activemask(), nwin);
#endif
    ext_identity(acc);
    // Straus pass over the two per-lane tables: four doublings and two additions per window as ONE straight-line
    // body (~150 KB of SASS) that the instruction prefetcher can follow; rolled into per-formula loops the same
    // work ran 1.4x slower (a fetch bubble per backward branch).  The B8 additions live in their own short loop.
    // What this kernel is most sensitive to is instruction supply: see the note on nwin above and
    // profiles/r1_ncu_icache_cliff.txt.
#pragma unroll 1
    for (int i = nwin - 1; i >= 0; i--) {
        if (i != nwin - 1) {
            ext_dbl<false>(acc, acc);
            ext_dbl<false>(acc, acc);
            ext_dbl<false>(acc, acc);
            ext_dbl<true>(acc, acc);
        }
        Niels nn;
        table_select(nn, tbl_a, park_digit4(park, 0, i));
        ext_add_niels<true>(acc, acc, nn);
        table_select(nn, tbl_r, park_digit4(park, 1, i));
        ext_add_niels_rt(acc, acc, nn, false, i == 0);      // T only where the B8 additions follow
    }
    // + w * B8: 16 signed 16-bit digits and the recoding carry against the fixed-base table, no doubling
#pragma unroll 1
    for (int k = BJJ_COMB_WINDOWS - 1; k >= 0; k--) {
        NielsAff nb;
        comb_select(nb, comb, k, park_digit16(park, 2, k));
        Niels nn;
        nn.ypx = nb.ypx;
        nn.ymx = nb.ymx;
        nn.t2d = nb.t2d;
        ext_add_niels_rt(acc, acc, nn, true, k != 0);
    }
    // acc == O = (0 : 1 : 1) ?   (Z != 0: complete formulas)
    return (fr_is_zero(acc.X) && fr_eq(acc.Y, acc.Z)) ? 1u : 0u;
}

// Exact lanes of verify: taken when R8 or A is not on the curve (the hash kernel has already stored hm).
// Every step whose inputs ARE curve points still yields the group element the reference computes
// (complete addition law), so only the off-curve parts replay the reference sequence:
//   l  = B8.mul_scalar(S)          B8 is on the curve            -> comb (same affine point)
//   kA = A.mul_scalar(8*hm)        A on the curve  (A_OFF = false) -> hm * (8A) by a table-free binary ladder
//                                  A off the curve (A_OFF = true)  -> literal LSB-first double-and-add
//                                                                      (src/lib.rs:149-164)
//   r  = R8 + kA, affine           literal add-2008-bbjlp + affine (Z == 0 -> (0,0)), src/lib.rs:407-411
// The two cases are queued separately so a warp never executes both ladders.
template <bool A_OFF>
BJJ_HD uint32_t verify_exact(const PointAff& r8, const uint32_t* s, const PointAff& a, const Fr& hm,
                             const CombEntry* comb, int mode) {
    PointAff l, ka, ra;
    PointExt accl;
    PointProj pl;
    fixed_base_comb(accl, comb, s);
    ext_to_proj(pl, accl);
    if (A_OFF) {
        proj_affine(l, pl);
        uint32_t k9[9];
        if (mode == BJJ_MODE_EDDSA) {
            k9[0] = hm.v[0] << 3;
#pragma unroll
            for (int i = 1; i < 8; i++) k9[i] = (hm.v[i] << 3) | (hm.v[i - 1] >> 29);
            k9[8] = hm.v[7] >> 29;
        } else {
#pragma unroll
            for (int i = 0; i < 8; i++) k9[i] = hm.v[i];
            k9[8] = 0;
        }
        mul_scalar_exact(ka, a, k9, 9);
    } else {
        PointExt p8, acc;
        ext_from_affine(p8, a);
        if (mode == BJJ_MODE_EDDSA) {
            ext_dbl<false>(p8, p8);
            ext_dbl<false>(p8, p8);
            ext_dbl<true>(p8, p8);
        }
        Niels n8;
        niels_from_ext(n8, p8);
        ext_identity(acc);
#pragma unroll 1
        for (int i = 253; i >= 0; i--) {      // hm < Q < 2^254
            ext_dbl<true>(acc, acc);
            if ((hm.v[i >> 5] >> (i & 31)) & 1) ext_add_niels<false>(acc, acc, n8);
        }
        PointProj pk;
        ext_to_proj(pk, acc);
        // both Z are non-zero (complete formulas on curve points): one shared inversion
        Fr t, ti, zl, zk;
        fr_mul(t, pl.z, pk.z);
        fr_inv(ti, t);
        fr_mul(zl, ti, pk.z);
        fr_mul(zk, ti, pl.z);
        fr_mul(l.x, pl.x, zl);
        fr_mul(l.y, pl.y, zl);
        fr_mul(ka.x, pk.x, zk);
        fr_mul(ka.y, pk.y, zk);
    }
    PointProj pr, pk2, sum;
    pr.x = r8.x;
    pr.y = r8.y;
    pr.z = fr_const(BJJ_ONE_M);
    pk2.x = ka.x;
    pk2.y = ka.y;
    pk2.z = fr_const(BJJ_ONE_M);
    proj_add_bbjlp(sum, pr, pk2);
    proj_affine(ra, sum);
    return (fr_eq(l.x, ra.x) && fr_eq(l.y, ra.y)) ? 1u : 0u;
}

// verify runs as a short pipeline of kernels so that no kernel carries another phase's registers or code:
//   phase 1 (lane_verify_hash): msg range check, on-curve gate (exact lanes are queued), hm = Poseidon(..)
//                               -> hm[i] (canonical integer), ok[i] = BJJ_OK_PENDING
//   phase 2 (lane_verify_ec):   Straus pass for the pending lanes -> ok[i] in {0, 1}
//   phase 3 (lane_verify_exact, other kernel): the queued off-curve lanes.
// `skip` (may be null): lanes whose decompression failed (verify_compressed) are rejected up front.
#define BJJ_OK_PENDING 2
// hm_out: 4 planes of `plane` 32-byte elements: hm | u | v (sign in bit 255) | w.
// S of lane i sits at 32-byte element index i * s_stride + s_off (1, 0 for a plain S array; 2, 1 inside sig64).
BJJ_HD void lane_verify_hash(const uint8_t* r8x, const uint8_t* r8y, const uint8_t* ax, const uint8_t* ay,
                             const uint8_t* msg32, const uint8_t* s_base, size_t s_stride, size_t s_off,
                             const uint8_t* skip, uint8_t* hm_out, size_t plane, uint8_t* ok, size_t i,
                             bool gate, const ExactQueue& qa, const ExactQueue& qr, uint32_t& flags, int mode,
                             bool split, uint8_t* msg_status) {
    if (skip && skip[i]) {
        ok[i] = 0;
        return;
    }
    uint32_t msg[8];
    load_u256(msg, msg32, i);
    const uint32_t qq[8] = BJJ_LIMBS8(BJJ_Q);
    const bool msg_bad = u256_lt(qq, msg);
    // verify: msg > Q -> false (src/lib.rs:396); verify_schnorr: Err("msg outside the Finite Field") (:365-367)
    if (msg_status) msg_status[i] = msg_bad ? (uint8_t)BJJ_ST_MSG_RANGE : (uint8_t)BJJ_ST_OK;
    if (msg_bad) {     // msg == Q is accepted and hashed as 0 (src/lib.rs:396-399)
        ok[i] = 0;
        return;
    }
    PointAff r8, a;
    load_fr(r8.x, r8x, i, flags);
    load_fr(r8.y, r8y, i, flags);
    load_fr(a.x, ax, i, flags);
    load_fr(a.y, ay, i, flags);
    uint32_t state = BJJ_OK_PENDING;
    if (gate) {
        // off-curve lanes are queued for the exact kernels (by case, so their warps do not diverge)
        if (!on_curve(a)) {
            exact_push(qa, i);
            state = 0;
        } else if (!on_curve(r8)) {
            exact_push(qr, i);
            state = 0;
        }
    }
    Fr mraw, mm, hm;
    fr_set(mraw, msg);
    fr_to_mont(mm, mraw);
    verify_hm(hm, r8, a, mm, mode);
    store_u256(hm_out, i, hm.v);
    ok[i] = (uint8_t)state;
    // scalars of the Straus pass: full width here (u = hm, v = 1, w = S); lane_verify_split shortens them
    if (state != BJJ_OK_PENDING || (split && mode == BJJ_MODE_EDDSA)) return;
    uint32_t sv[8], one[8];
    load_u256(sv, s_base, i * s_stride + s_off);
#pragma unroll
    for (int k = 0; k < 8; k++) one[k] = k == 0 ? 1u : 0u;
    store_u256(hm_out, plane + i, hm.v);
    store_u256(hm_out, 2 * plane + i, one);
    store_u256(hm_out, 3 * plane + i, sv);
}

// test hook (bjj_split_scalars_batch): the split on caller-supplied h and s
BJJ_HD void lane_split_scalars(const uint8_t* h32, const uint8_t* s32, uint8_t* u32, uint8_t* v32, uint8_t* w32, size_t i) {
    uint32_t h[8], sv[8], u[8], v[8], w[8], vneg = 0;
    load_u256(h, h32, i);
    load_u256(sv, s32, i);
    split_scalars(u, v, vneg, h);
    split_scale_s(w, sv, v);
    v[7] |= vneg << 31;
    store_u256(u32, i, u);
    store_u256(v32, i, v);
    store_u256(w32, i, w);
}

// phase 1b (EdDSA): half-size scalars for the pending lanes (split.cuh).  Its own kernel: integer-ALU work with
// lane-dependent trip counts, which inside the hash kernel would leave that kernel's warps out of step.
BJJ_HD void lane_verify_split(const uint8_t* s_base, size_t s_stride, size_t s_off, uint8_t* hm_io, size_t plane,
                              const uint8_t* ok, size_t i) {
    if (ok[i] != BJJ_OK_PENDING) return;
    uint32_t hm[8], sv[8], u[8], v[8], w[8], vneg = 0;
    load_u256(hm, hm_io, i);
    load_u256(sv, s_base, i * s_stride + s_off);
    split_scalars(u, v, vneg, hm);
    split_scale_s(w, sv, v);
    v[7] |= vneg << 31;
    store_u256(hm_io, plane + i, u);
    store_u256(hm_io, 2 * plane + i, v);
    store_u256(hm_io, 3 * plane + i, w);
}

BJJ_HD void lane_verify_ec(const uint8_t* r8x, const uint8_t* r8y, const uint8_t* ax, const uint8_t* ay,
                           const uint8_t* hm_in, size_t plane, uint8_t* ok, size_t i, const LaneTable& tbl_a,
                           const LaneTable& tbl_r, const CombEntry* comb, int mode, const ScalarPark& park) {
    if (ok[i] != BJJ_OK_PENDING) return;
    uint32_t flags = 0;
    PointAff r8, a;
    VerifyScalars sc;
    load_u256(sc.u, hm_in, plane + i);
    load_u256(sc.v, hm_in, 2 * plane + i);
    load_u256(sc.w, hm_in, 3 * plane + i);
    sc.vneg = sc.v[7] >> 31;
    sc.v[7] &= 0x7FFFFFFFu;
    load_fr(r8.x, r8x, i, flags);
    load_fr(r8.y, r8y, i, flags);
    load_fr(a.x, ax, i, flags);
    load_fr(a.y, ay, i, flags);
    ok[i] = (uint8_t)verify_fast(r8, a, sc, tbl_a, tbl_r, comb, mode, park);
}

template <bool A_OFF>
BJJ_HD void lane_verify_exact(const uint8_t* r8x, const uint8_t* r8y, const uint8_t* s32, const uint8_t* ax,
                              const uint8_t* ay, const uint8_t* hm_in, uint8_t* ok, size_t i, const CombEntry* comb,
                              int mode) {
    uint32_t s[8], flags = 0;
    PointAff r8, a;
    Fr hm;
    load_u256(s, s32, i);
    load_u256(hm.v, hm_in, i);
    load_fr(r8.x, r8x, i, flags);
    load_fr(r8.y, r8y, i, flags);
    load_fr(a.x, ax, i, flags);
    load_fr(a.y, ay, i, flags);
    ok[i] = (uint8_t)verify_exact<A_OFF>(r8, s, a, hm, comb, mode);
}

}  // namespace bjj
