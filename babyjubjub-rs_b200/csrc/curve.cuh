// BabyJubJub point arithmetic.
//
// Two families of formulas live here:
//
//  (1) LITERAL: the reference's own projective add-2008-bbjlp (src/lib.rs:88-131), its affine()
//      (src/lib.rs:70-85, Z == 0 -> (0,0)) and its LSB-first double-and-add (src/lib.rs:149-164).
//      Needed for bit-exact *projective* outputs (add_batch) and for lanes whose input point is NOT
//      on the curve: there the formulas are no group law and the result depends on the exact
//      operation order, so those lanes replay the reference sequence ("exact lane").
//
//  (2) FAST: for on-curve inputs the result is a group element, so any correct algorithm gives the
//      same canonical affine coordinates.  We move to the isomorphic a = -1 curve
//          x' = sqrt(-a) * x :   -x'^2 + y^2 = 1 + d' x'^2 y^2,   d' = -d/a   (d' non-square, so
//      the unified extended-coordinate formulas are complete), and use
//          dbl  : 4S + 3M (+1M when T is wanted)        [dbl-2008-hwcd, a = -1]
//          add  : 8M against a cached (Y+X, Y-X, 2d'T, 2Z) entry, 7M when Z2 = 1   [add-2008-hwcd-3]
#pragma once
#include "fr.cuh"

namespace bjj {

struct PointAff {   // Montgomery-form affine point on the ORIGINAL curve (reference `Point`, src/lib.rs:135-138)
    Fr x, y;
};
struct PointProj {  // reference `PointProjective`, src/lib.rs:63-67
    Fr x, y, z;
};
struct PointExt {   // extended coordinates on the a = -1 curve
    Fr X, Y, Z, T;
};
struct Niels {      // cached addend on the a = -1 curve: (Y+X, Y-X, 2d'T, 2Z)
    Fr ypx, ymx, t2d, z2;
};
struct NielsAff {   // cached affine addend (Z = 1): (y+x, y-x, 2d'xy)
    Fr ypx, ymx, t2d;
};

// ---------------------------------------------------------------------------------------------
// (1) literal reference formulas
// ---------------------------------------------------------------------------------------------

// PointProjective::add -- add-2008-bbjlp exactly as src/lib.rs:88-131 sequences it (13 fmul).
BJJ_HD void proj_add_bbjlp(PointProj& r, const PointProj& p, const PointProj& q) {
    const Fr cA = fr_const(BJJ_A_M), cD = fr_const(BJJ_D_M);
    Fr a, b, c, d, e, f, g, aux, t, x3, y3, z3;
    fr_mul(a, p.z, q.z);
    fr_sqr(b, a);
    fr_mul(c, p.x, q.x);
    fr_mul(d, p.y, q.y);
    fr_mul(e, cD, c);
    fr_mul(e, e, d);
    fr_sub(f, b, e);
    fr_add(g, b, e);
    fr_add(aux, p.x, p.y);
    fr_add(t, q.x, q.y);
    fr_mul(aux, aux, t);
    fr_sub(aux, aux, c);
    fr_sub(aux, aux, d);
    fr_mul(x3, a, f);
    fr_mul(x3, x3, aux);
    fr_mul(t, cA, c);
    fr_sub(t, d, t);
    fr_mul(y3, a, g);
    fr_mul(y3, y3, t);
    fr_mul(z3, f, g);
    r.x = x3;
    r.y = y3;
    r.z = z3;
}

// PointProjective::affine (src/lib.rs:70-85): Z == 0 -> (0, 0).  Fermat inverse per lane.
BJJ_HD void proj_affine(PointAff& r, const PointProj& p) {
    if (fr_is_zero(p.z)) {
        fr_zero(r.x);
        fr_zero(r.y);
        return;
    }
    Fr zi;
    fr_inv(zi, p.z);
    fr_mul(r.x, p.x, zi);
    fr_mul(r.y, p.y, zi);
}

// ---------------------------------------------------------------------------------------------
// (2) fast path on the a = -1 model
// ---------------------------------------------------------------------------------------------

// a*x^2 + y^2 == 1 + d*x^2*y^2   (the curve equation behind src/lib.rs:29-31)
BJJ_HD bool on_curve(const PointAff& p) {
    const Fr cA = fr_const(BJJ_A_M), cD = fr_const(BJJ_D_M), one = fr_const(BJJ_ONE_M);
    Fr x2, y2, l, r;
    fr_sqr(x2, p.x);
    fr_sqr(y2, p.y);
    fr_mul(l, cA, x2);
    fr_add(l, l, y2);
    fr_mul(r, x2, y2);
    fr_mul(r, r, cD);
    fr_add(r, r, one);
    return fr_eq(l, r);
}

BJJ_HD void ext_identity(PointExt& p) {
    fr_zero(p.X);
    p.Y = fr_const(BJJ_ONE_M);
    p.Z = fr_const(BJJ_ONE_M);
    fr_zero(p.T);
}

// original-curve affine -> a = -1 extended
BJJ_HD void ext_from_affine(PointExt& r, const PointAff& p) {
    const Fr s = fr_const(BJJ_SQRT_NEG_A_M);
    fr_mul(r.X, p.x, s);
    r.Y = p.y;
    r.Z = fr_const(BJJ_ONE_M);
    fr_mul(r.T, r.X, r.Y);
}

// r = 2p.  WANT_T = false skips the T3 product (next op is another doubling).
template <bool WANT_T>
BJJ_HD void ext_dbl(PointExt& r, const PointExt& p) {
    Fr xx, yy, zz2, s, e, g, f, h;
    fr_sqr(xx, p.X);
    fr_sqr(yy, p.Y);
    fr_sqr(zz2, p.Z);
    fr_dbl(zz2, zz2);
    fr_add(s, p.X, p.Y);
    fr_sqr(s, s);
    fr_add(h, yy, xx);     // H' = Y^2 + X^2
    fr_sub(g, yy, xx);     // G  = Y^2 - X^2
    fr_sub(e, s, h);       // E  = 2XY
    fr_sub(f, zz2, g);     // F' = 2Z^2 - G
    fr_mul(r.X, e, f);
    fr_mul(r.Y, h, g);
    fr_mul(r.Z, g, f);
    if (WANT_T) fr_mul(r.T, e, h);
}

BJJ_HD void niels_from_ext(Niels& n, const PointExt& p) {
    const Fr d2 = fr_const(BJJ_TWO_DP_M);
    fr_add(n.ypx, p.Y, p.X);
    fr_sub(n.ymx, p.Y, p.X);
    fr_mul(n.t2d, p.T, d2);
    fr_dbl(n.z2, p.Z);
}

BJJ_HD void niels_identity(Niels& n) {
    n.ypx = fr_const(BJJ_ONE_M);
    n.ymx = fr_const(BJJ_ONE_M);
    fr_zero(n.t2d);
    fr_dbl(n.z2, n.ypx);
}

// -n : swap (Y+X, Y-X), negate 2d'T
BJJ_HD void niels_cneg(Niels& n, bool neg) {
    Fr nt;
    fr_neg(nt, n.t2d);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint32_t a = n.ypx.v[i], b = n.ymx.v[i];
        n.ypx.v[i] = neg ? b : a;
        n.ymx.v[i] = neg ? a : b;
        n.t2d.v[i] = neg ? nt.v[i] : n.t2d.v[i];
    }
}
BJJ_HD void niels_aff_cneg(NielsAff& n, bool neg) {
    Fr nt;
    fr_neg(nt, n.t2d);
#pragma unroll
    for (int i = 0; i < 8; i++) {
        uint32_t a = n.ypx.v[i], b = n.ymx.v[i];
        n.ypx.v[i] = neg ? b : a;
        n.ymx.v[i] = neg ? a : b;
        n.t2d.v[i] = neg ? nt.v[i] : n.t2d.v[i];
    }
}

// r = p + n   (8M; 7M for T-less output)
template <bool WANT_T>
BJJ_HD void ext_add_niels(PointExt& r, const PointExt& p, const Niels& n) {
    Fr a, b, c, d, e, f, g, h, t;
    fr_add(t, p.Y, p.X);
    fr_mul(a, t, n.ypx);
    fr_sub(t, p.Y, p.X);
    fr_mul(b, t, n.ymx);
    fr_mul(c, p.T, n.t2d);
    fr_mul(d, p.Z, n.z2);
    fr_sub(e, a, b);
    fr_add(h, a, b);
    fr_add(g, d, c);
    fr_sub(f, d, c);
    fr_mul(r.X, e, f);
    fr_mul(r.Y, g, h);
    fr_mul(r.Z, f, g);
    if (WANT_T) fr_mul(r.T, e, h);
}

// r = p + n with Z(n) = 1   (7M; 6M for T-less output)
template <bool WANT_T>
BJJ_HD void ext_add_niels_aff(PointExt& r, const PointExt& p, const NielsAff& n) {
    Fr a, b, c, d, e, f, g, h, t;
    fr_add(t, p.Y, p.X);
    fr_mul(a, t, n.ypx);
    fr_sub(t, p.Y, p.X);
    fr_mul(b, t, n.ymx);
    fr_mul(c, p.T, n.t2d);
    fr_dbl(d, p.Z);
    fr_sub(e, a, b);
    fr_add(h, a, b);
    fr_add(g, d, c);
    fr_sub(f, d, c);
    fr_mul(r.X, e, f);
    fr_mul(r.Y, g, h);
    fr_mul(r.Z, f, g);
    if (WANT_T) fr_mul(r.T, e, h);
}

// Run-time flavours of the formulas above, for the short loops around the Straus pass (table set-up, B8
// additions) that keep ONE copy of a formula in the instruction stream: a fully inlined field multiplication is
// ~3 KB of SASS.  The hot window body itself stays straight-line (see verify_fast).
BJJ_HD void ext_dbl_rt(PointExt& r, const PointExt& p, bool want_t) {
    Fr xx, yy, zz2, s, e, g, f, h;
    fr_sqr(xx, p.X);
    fr_sqr(yy, p.Y);
    fr_sqr(zz2, p.Z);
    fr_dbl(zz2, zz2);
    fr_add(s, p.X, p.Y);
    fr_sqr(s, s);
    fr_add(h, yy, xx);
    fr_sub(g, yy, xx);
    fr_sub(e, s, h);
    fr_sub(f, zz2, g);
    fr_mul(r.X, e, f);
    fr_mul(r.Y, h, g);
    fr_mul(r.Z, g, f);
    if (want_t) fr_mul(r.T, e, h);
}
// r = p + n; `affine`: Z(n) = 1 (n.z2 is not read)
BJJ_HD void ext_add_niels_rt(PointExt& r, const PointExt& p, const Niels& n, bool affine, bool want_t) {
    Fr a, b, c, d, e, f, g, h, t;
    fr_add(t, p.Y, p.X);
    fr_mul(a, t, n.ypx);
    fr_sub(t, p.Y, p.X);
    fr_mul(b, t, n.ymx);
    fr_mul(c, p.T, n.t2d);
    if (affine) {
        fr_dbl(d, p.Z);
    } else {
        fr_mul(d, p.Z, n.z2);
    }
    fr_sub(e, a, b);
    fr_add(h, a, b);
    fr_add(g, d, c);
    fr_sub(f, d, c);
    fr_mul(r.X, e, f);
    fr_mul(r.Y, g, h);
    fr_mul(r.Z, f, g);
    if (want_t) fr_mul(r.T, e, h);
}

// a = -1 extended -> projective point on the ORIGINAL curve: (X / sqrt(-a) : Y : Z)
BJJ_HD void ext_to_proj(PointProj& r, const PointExt& p) {
    const Fr si = fr_const(BJJ_INV_SQRT_NEG_A_M);
    fr_mul(r.x, p.X, si);
    r.y = p.Y;
    r.z = p.Z;
}

// ---------------------------------------------------------------------------------------------
// scalar recoding
// ---------------------------------------------------------------------------------------------

// Signed radix-16: n = sum_{i<64} d_i 16^i + c 16^64 with d_i in [-8, 7], c in {0,1}.
// Computed as n' = n + 0x88..8 (carry-out c); d_i = nibble_i(n') - 8.
struct Recode4 {
    uint32_t w[8];
    uint32_t top;
};
BJJ_HD void recode4(Recode4& rc, const uint32_t* n) {
    uint32_t eights[8];
#pragma unroll
    for (int i = 0; i < 8; i++) eights[i] = 0x88888888u;
    rc.top = add256(rc.w, n, eights);
}
BJJ_HD int recode4_digit(const Recode4& rc, int i) {   // i in [0, 64)
    return (int)((rc.w[i >> 3] >> ((i & 7) * 4)) & 15u) - 8;
}

// Signed radix-2^16: n = sum_{i<16} d_i 65536^i + c 65536^16, d_i in [-32768, 32767].
struct Recode16 {
    uint32_t w[8];
    uint32_t top;
};
BJJ_HD void recode16(Recode16& rc, const uint32_t* n) {
    uint32_t off[8];
#pragma unroll
    for (int i = 0; i < 8; i++) off[i] = 0x80008000u;
    rc.top = add256(rc.w, n, off);
}
BJJ_HD int recode16_digit(const Recode16& rc, int i) {   // i in [0, 16)
    return (int)((rc.w[i >> 1] >> ((i & 1) * 16)) & 65535u) - 32768;
}

// Signed radix-2^8: n = sum_{i<32} d_i 256^i + c 256^32, d_i in [-128, 127], c in {0, 1}.
struct Recode8 {
    uint32_t w[8];
    uint32_t top;
};
BJJ_HD void recode8(Recode8& rc, const uint32_t* n) {
    uint32_t off[8];
#pragma unroll
    for (int i = 0; i < 8; i++) off[i] = 0x80808080u;
    rc.top = add256(rc.w, n, off);
}
BJJ_HD int recode8_digit(const Recode8& rc, int i) {   // i in [0, 32)
    return (int)((rc.w[i >> 2] >> ((i & 3) * 8)) & 255u) - 128;
}

}  // namespace bjj
