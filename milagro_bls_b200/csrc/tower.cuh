// Extension tower Fp2 -> Fp6 -> Fp12 (2-3-2) for BLS12-381.
//
//   Fp2  = Fp[i]/(i^2+1)            Fp6 = Fp2[v]/(v^3 - xi), xi = 1+i           Fp12 = Fp6[w]/(w^2 - v)
//
// so an Fp12 element is sum_{k=0..5} f_k w^k with f_k in Fp2 and w^6 = xi:
//   c0 = (w^0, w^2, w^4), c1 = (w^1, w^3, w^5).
// The reference uses a 2-2-3 tower (/root/reference/incubator-milagro-crypto-rust/src/fp4.rs,
// fp12.rs:300-366: Fp12 = Fp4[w]/(w^3-j), j^2 = 1+i) which holds the same six Fp2 coefficients; its wire
// order (fp12.rs:859-913) is w^0, w^3, w^1, w^4, w^2, w^5 -- see fp12_to_wire() (SURVEY.md B.2).
#pragma once
#include "fp.cuh"

// The Fp6 / Fp12 layers are templates over the Fp2 representation F2: fp2 (one thread per value; fp6 / fp12 below) or
// fp2h (lane pairs, fp2h.cuh) -- the same way the point formulas of curve.cuh / pairing.cuh are.
template <class F2>
struct fp6_t {
    F2 c0, c1, c2;
};
template <class F2>
struct fp12_t {
    fp6_t<F2> c0, c1;
};
typedef fp6_t<fp2> fp6;
typedef fp12_t<fp2> fp12;

// ---------------------------------------------------------------- Fp2
B3_FN void fp2_add(fp2& r, const fp2& a, const fp2& b) { fp_add(r.c0, a.c0, b.c0); fp_add(r.c1, a.c1, b.c1); }
B3_FN void fp2_sub(fp2& r, const fp2& a, const fp2& b) { fp_sub(r.c0, a.c0, b.c0); fp_sub(r.c1, a.c1, b.c1); }
B3_FN void fp2_neg(fp2& r, const fp2& a) { fp_neg(r.c0, a.c0); fp_neg(r.c1, a.c1); }
B3_FN void fp2_dbl(fp2& r, const fp2& a) { fp_dbl(r.c0, a.c0); fp_dbl(r.c1, a.c1); }
B3_FN void fp2_half(fp2& r, const fp2& a) { fp_half(r.c0, a.c0); fp_half(r.c1, a.c1); }
B3_FN void fp2_conj(fp2& r, const fp2& a) { r.c0 = a.c0; fp_neg(r.c1, a.c1); }
B3_FN bool fp2_is_zero(const fp2& a) { return fp_is_zero(a.c0) && fp_is_zero(a.c1); }
B3_FN bool fp2_eq(const fp2& a, const fp2& b) { return fp_eq(a.c0, b.c0) && fp_eq(a.c1, b.c1); }
B3_FN void fp2_select(fp2& r, bool c, const fp2& a, const fp2& b) { fp_select(r.c0, c, a.c0, b.c0); fp_select(r.c1, c, a.c1, b.c1); }
B3_FN void fp2_zero(fp2& r) { r.c0 = FP_NIL; r.c1 = FP_NIL; }
B3_FN void fp2_one(fp2& r) { r.c0 = FP_ONE; r.c1 = FP_NIL; }

// (a0 + a1 i)(b0 + b1 i) = (a0 b0 + (-a1) b1) + (a0 b1 + a1 b0) i: two dual products with one reduction each
// (2 x 444 multiply-accumulates, fp.cuh: fp_mul2_inl), both inlined into one by-value out-of-line routine.
B3_FN_NOINLINE fp2 fp2_mul_v(fp2 a, fp2 b) {
    fp2 r;
    fp na1;
    fp_neg_nr(na1, a.c1);
    fp_mul2_inl(r.c0, a.c0, b.c0, na1, b.c1);
    fp_mul2_inl(r.c1, a.c0, b.c1, a.c1, b.c0);
    return r;
}
B3_FN void fp2_mul(fp2& r, const fp2& a, const fp2& b) { r = fp2_mul_v(a, b); }
// (a0+a1)(a0-a1) + 2 a0 a1 i : 2 Fp mults
B3_FN_NOINLINE fp2 fp2_sqr_v(fp2 a) {
    fp2 r;
    fp s, d, m;
    fp_add_nr(s, a.c0, a.c1);             // < 4p: the first operand of the product
    fp_sub(d, a.c0, a.c1);
    fp_mul_inl(m, a.c0, a.c1);
    fp_mul_inl(r.c0, s, d);
    fp_dbl(r.c1, m);
    return r;
}
B3_FN void fp2_sqr(fp2& r, const fp2& a) { r = fp2_sqr_v(a); }
B3_FN void fp2_mul_fp(fp2& r, const fp2& a, const fp& s) { fp_mul(r.c0, a.c0, s); fp_mul(r.c1, a.c1, s); }
// * xi = (1+i)
B3_FN void fp2_mul_xi(fp2& r, const fp2& a) {
    fp t;
    fp_sub(t, a.c0, a.c1);
    fp_add(r.c1, a.c0, a.c1);
    r.c0 = t;
}
B3_FN void fp2_mul3(fp2& r, const fp2& a) { fp2 t; fp2_dbl(t, a); fp2_add(r, t, a); }
// 1/a = conj(a)/N(a);  0 -> 0
B3_FN_NOINLINE void fp2_inv(fp2& r, const fp2& a) {
    fp n, t;
    fp_sqr(n, a.c0);
    fp_sqr(t, a.c1);
    fp_add(n, n, t);
    fp_inv(n, n);
    fp_mul(r.c0, a.c0, n);
    fp_mul(t, a.c1, n);
    fp_neg(r.c1, t);
}
// RFC 9380 sgn0 for m = 2 (= reference A/fp2.rs:449-455); input in Montgomery form
B3_FN_NOINLINE uint32_t fp2_sgn0(const fp2& a) {
    fp r0, r1;
    fp_from_mont(r0, a.c0);
    fp_from_mont(r1, a.c1);
    uint32_t s0 = r0.l[0] & 1u, z0 = fp_is_zero(r0) ? 1u : 0u, s1 = r1.l[0] & 1u;
    return s0 | (z0 & s1);
}

// Square root in Fp2 with two Fp exponentiations (norm trick, p = 3 mod 4).
//   Let n = N(a) = a0^2 + a1^2.  a is a square in Fp2 iff n is a square in Fp.
//   If not, returns false and a root of zmul*a where N(zmul) = 5 (zmul = SSWU Z = -(2+i)) is produced
//   from the same exponentiation: sqrt(5 n) = sqrt(-5) * sqrt(-n).
//   root = x0 + x1 i with x0^2 = (a0 + s)/2 or x1^2 = ..., handled by the chi trick of fp_sqrt_ratio_parts.
// out: r = sqrt(a) if a is square, else sqrt(Z * a).  Which of the two roots is unspecified.
B3_FN_NOINLINE bool fp2_sqrt_or_z(fp2& r, const fp2& a) {
    fp n, t, s, sinv;
    fp_sqr(n, a.c0);
    fp_sqr(t, a.c1);
    fp_add(n, n, t);
    bool sq = fp_sqrt_ratio_parts(s, sinv, n);          // s^2 = n (sq) or s^2 = -n (!sq)
    fp2 b;
    if (sq) {
        b = a;
    } else {
        fp2_mul(b, a, SSWU_Z);                           // N(b) = 5 n, sqrt = sqrt(-5) * s
        fp_mul(s, s, FP_SQRT_M5);
    }
    // now s^2 = N(b), b = b0 + b1 i.  delta = (b0 + s)/2; exactly one of delta, (b0 - s)/2 is a QR
    // unless b1 == 0.
    fp delta, x, xinv;
    fp_add(delta, b.c0, s);
    fp_half(delta, delta);
    if (fp_is_zero(delta)) {                             // b0 = -s: then b1 = 0 and b = -|..|; use other branch
        fp_sub(delta, b.c0, s);
        fp_half(delta, delta);
    }
    bool dq = fp_sqrt_ratio_parts(x, xinv, delta);       // x^2 = +-delta, xinv = 1/x
    // y = b1 / (2x)
    fp y, hb1;
    fp_half(hb1, b.c1);
    fp_mul(y, hb1, xinv);
    if (dq) {                                            // x^2 = delta: root = x + y i
        r.c0 = x; r.c1 = y;
    } else {                                             // x^2 = -delta: (y + ... ) root = y - x i ... see below
        // (x0 + x1 i)^2 = b with x0^2 = delta_minus.  delta_minus = -b1^2/(4 delta) = (b1/(2x))^2 = y^2,
        // so x0 = y and x1 = b1/(2 x0) = b1/(2y) = x^2 * ... = -delta*2/b1 ... use x1 = b1 * x /(2 * x^2 * y)
        // simpler: x1 = b1/(2y) and y = b1/(2x) => x1 = x.  Check sign: (y + x i)^2 = y^2 - x^2 + 2xy i
        //   = delta_minus + delta + b1 i = b0 + b1 i.
        r.c0 = y; r.c1 = x;
    }
    return sq;
}

// Square root of a RATIO u / v in Fp2 (v != 0) with two Fp exponentiations and no inversion:
//   r = sqrt(u / v)       and returns true   if u / v is a square in Fp2,
//   r = sqrt(Z u / v)     and returns false  otherwise  (Z = SSWU_Z, N(Z) = 5).
// Method: X = u / v = W / b with W = u conj(v), b = N(v) in Fp.  N(X) = N(W) / b^2, so  s = sqrt(N(X)) = t / b with
// t = sqrt(N(W)) (first exponentiation; if N(W) is a non-residue switch to Z W, t <- sqrt(-5) t as in fp2_sqrt_or_z).
// With D = (W0 + t) / 2 = b delta:  x0 = sqrt(delta) = sqrt(D / b) = D b g,  g = (D b^3)^((p-3)/4)  (second
// exponentiation), chi = g^2 D b^3 = +-1, and 1 / (b x0) = chi g b, so the other coordinate W1 / (2 b x0) needs no
// inversion either.  chi = -1 means x0^2 = -delta and the two coordinates swap roles (see fp2_sqrt_or_z).
B3_FN_NOINLINE bool fp2_sqrt_ratio_or_z(fp2& r, const fp2& u, const fp2& v) {
    fp b, n, t, tinv, s0;
    fp2 W, cv;
    fp_sqr(b, v.c0);
    fp_sqr(s0, v.c1);
    fp_add(b, b, s0);                                    // b = N(v)
    fp2_conj(cv, v);
    fp2_mul(W, u, cv);                                   // W = u conj(v)
    fp_sqr(n, W.c0);
    fp_sqr(s0, W.c1);
    fp_add(n, n, s0);                                    // N(W)
    bool sq = fp_sqrt_ratio_parts(t, tinv, n);           // t^2 = N(W) (sq) or -N(W) (!sq)
    if (!sq) {
        fp2_mul(W, W, SSWU_Z);                           // N(Z W) = 5 N(W), sqrt = sqrt(-5) t
        fp_mul(t, t, FP_SQRT_M5);
    }
    fp D;
    fp_add(D, W.c0, t);
    fp_half(D, D);
    if (fp_is_zero(D)) {                                 // W0 = -t: W1 = 0; use the conjugate branch
        fp_sub(D, W.c0, t);
        fp_half(D, D);
    }
    fp b2, b3, E, g, chi, x0, yv, hw1;
    fp_sqr(b2, b);
    fp_mul(b3, b2, b);
    fp_mul(E, D, b3);
    fp_pow_const(g, E, FP_EXP_SQRT_G);                   // g = E^((p-3)/4)
    fp_mul(chi, g, E);
    fp_mul(chi, chi, g);                                 // chi = E^((p-1)/2) in {0, 1, -1}
    bool plus = !fp_eq(chi, FP_M_ONE);
    fp_mul(x0, D, b);
    fp_mul(x0, x0, g);                                   // x0 = D b g,  x0^2 = chi D / b
    fp_half(hw1, W.c1);
    fp_mul(yv, hw1, b);
    fp_mul(yv, yv, g);                                   // (W1 / 2) b g
    fp nyv;
    fp_neg(nyv, yv);
    if (plus) { r.c0 = x0; r.c1 = yv; }
    else { r.c0 = nyv; r.c1 = x0; }
    return sq;
}

// a constant of Fp2 in the representation F2 (the lane-pair overload picks this lane's half, fp2h.cuh)
B3_FN void f2_const(fp2& r, const fp2& c) { r = c; }

// ---------------------------------------------------------------- Fp6
template <class F2>
B3_FN void fp6_add(fp6_t<F2>& r, const fp6_t<F2>& a, const fp6_t<F2>& b) { fp2_add(r.c0, a.c0, b.c0); fp2_add(r.c1, a.c1, b.c1); fp2_add(r.c2, a.c2, b.c2); }
template <class F2>
B3_FN void fp6_sub(fp6_t<F2>& r, const fp6_t<F2>& a, const fp6_t<F2>& b) { fp2_sub(r.c0, a.c0, b.c0); fp2_sub(r.c1, a.c1, b.c1); fp2_sub(r.c2, a.c2, b.c2); }
template <class F2>
B3_FN void fp6_neg(fp6_t<F2>& r, const fp6_t<F2>& a) { fp2_neg(r.c0, a.c0); fp2_neg(r.c1, a.c1); fp2_neg(r.c2, a.c2); }
// * v : (c0, c1, c2) -> (xi c2, c0, c1)
template <class F2>
B3_FN void fp6_mul_v(fp6_t<F2>& r, const fp6_t<F2>& a) {
    F2 t;
    fp2_mul_xi(t, a.c2);
    r.c2 = a.c1;
    r.c1 = a.c0;
    r.c0 = t;
}
template <class F2>
B3_FN_NOINLINE void fp6_mul(fp6_t<F2>& r, const fp6_t<F2>& a, const fp6_t<F2>& b) {
    F2 v0, v1, v2, t0, t1, t2;
    fp2_mul(v0, a.c0, b.c0);
    fp2_mul(v1, a.c1, b.c1);
    fp2_mul(v2, a.c2, b.c2);
    // c0 = v0 + xi((a1+a2)(b1+b2) - v1 - v2)
    fp2_add(t0, a.c1, a.c2);
    fp2_add(t1, b.c1, b.c2);
    fp2_mul(t0, t0, t1);
    fp2_sub(t0, t0, v1);
    fp2_sub(t0, t0, v2);
    fp2_mul_xi(t0, t0);
    fp2_add(t0, t0, v0);
    // c1 = (a0+a1)(b0+b1) - v0 - v1 + xi v2
    fp2_add(t1, a.c0, a.c1);
    fp2_add(t2, b.c0, b.c1);
    fp2_mul(t1, t1, t2);
    fp2_sub(t1, t1, v0);
    fp2_sub(t1, t1, v1);
    fp2_mul_xi(t2, v2);
    fp2_add(t1, t1, t2);
    // c2 = (a0+a2)(b0+b2) - v0 - v2 + v1
    F2 u0, u1;
    fp2_add(u0, a.c0, a.c2);
    fp2_add(u1, b.c0, b.c2);
    fp2_mul(u0, u0, u1);
    fp2_sub(u0, u0, v0);
    fp2_sub(u0, u0, v2);
    fp2_add(r.c2, u0, v1);
    r.c0 = t0;
    r.c1 = t1;
}
template <class F2>
B3_FN void fp6_sqr(fp6_t<F2>& r, const fp6_t<F2>& a) { fp6_mul(r, a, a); }
// a * (b0, 0, 0)
template <class F2>
B3_FN void fp6_mul_fp2(fp6_t<F2>& r, const fp6_t<F2>& a, const F2& b0) {
    fp2_mul(r.c0, a.c0, b0); fp2_mul(r.c1, a.c1, b0); fp2_mul(r.c2, a.c2, b0);
}
// a * (0, b1, b2)
template <class F2>
B3_FN_NOINLINE void fp6_mul_by_12(fp6_t<F2>& r, const fp6_t<F2>& a, const F2& b1, const F2& b2) {
    F2 v1, v2, t0, t1, t2;
    fp2_mul(v1, a.c1, b1);
    fp2_mul(v2, a.c2, b2);
    // c0 = xi (a1 b2 + a2 b1) = xi((a1+a2)(b1+b2) - v1 - v2)
    fp2_add(t0, a.c1, a.c2);
    fp2_add(t1, b1, b2);
    fp2_mul(t0, t0, t1);
    fp2_sub(t0, t0, v1);
    fp2_sub(t0, t0, v2);
    fp2_mul_xi(t0, t0);
    // c1 = a0 b1 + xi v2 ; c2 = a0 b2 + v1
    fp2_mul(t1, a.c0, b1);
    fp2_mul_xi(t2, v2);
    fp2_add(t1, t1, t2);
    fp2_mul(t2, a.c0, b2);
    fp2_add(r.c2, t2, v1);
    r.c0 = t0;
    r.c1 = t1;
}
template <class F2>
B3_FN_NOINLINE void fp6_inv(fp6_t<F2>& r, const fp6_t<F2>& a) {
    F2 A, B, C, t, F;
    fp2_sqr(A, a.c0); fp2_mul(t, a.c1, a.c2); fp2_mul_xi(t, t); fp2_sub(A, A, t);      // a0^2 - xi a1 a2
    fp2_sqr(B, a.c2); fp2_mul_xi(B, B); fp2_mul(t, a.c0, a.c1); fp2_sub(B, B, t);      // xi a2^2 - a0 a1
    fp2_sqr(C, a.c1); fp2_mul(t, a.c0, a.c2); fp2_sub(C, C, t);                        // a1^2 - a0 a2
    fp2_mul(F, a.c0, A);
    fp2_mul(t, a.c2, B); fp2_mul_xi(t, t); fp2_add(F, F, t);
    fp2_mul(t, a.c1, C); fp2_mul_xi(t, t); fp2_add(F, F, t);
    fp2_inv(F, F);
    fp2_mul(r.c0, A, F); fp2_mul(r.c1, B, F); fp2_mul(r.c2, C, F);
}

// ---------------------------------------------------------------- Fp12
template <class F2>
B3_FN void fp12_one(fp12_t<F2>& r) {
    fp2_one(r.c0.c0); fp2_zero(r.c0.c1); fp2_zero(r.c0.c2);
    fp2_zero(r.c1.c0); fp2_zero(r.c1.c1); fp2_zero(r.c1.c2);
}
template <class F2>
B3_FN bool fp12_eq(const fp12_t<F2>& a, const fp12_t<F2>& b) {
    return fp2_eq(a.c0.c0, b.c0.c0) && fp2_eq(a.c0.c1, b.c0.c1) && fp2_eq(a.c0.c2, b.c0.c2) &&
           fp2_eq(a.c1.c0, b.c1.c0) && fp2_eq(a.c1.c1, b.c1.c1) && fp2_eq(a.c1.c2, b.c1.c2);
}
template <class F2>
B3_FN bool fp12_is_one(const fp12_t<F2>& a) {
    F2 one;
    fp2_one(one);
    const bool e0 = fp2_eq(a.c0.c0, one), z1 = fp2_is_zero(a.c0.c1), z2 = fp2_is_zero(a.c0.c2);      // (lane pairs: every
    const bool z3 = fp2_is_zero(a.c1.c0), z4 = fp2_is_zero(a.c1.c1), z5 = fp2_is_zero(a.c1.c2);      //  test runs on both lanes)
    return e0 && z1 && z2 && z3 && z4 && z5;
}
template <class F2>
B3_FN_NOINLINE void fp12_mul(fp12_t<F2>& r, const fp12_t<F2>& a, const fp12_t<F2>& b) {
    fp6_t<F2> t0, t1, s0, s1;
    fp6_mul(t0, a.c0, b.c0);
    fp6_mul(t1, a.c1, b.c1);
    fp6_add(s0, a.c0, a.c1);
    fp6_add(s1, b.c0, b.c1);
    fp6_mul(s0, s0, s1);
    fp6_sub(s0, s0, t0);
    fp6_sub(r.c1, s0, t1);
    fp6_mul_v(t1, t1);
    fp6_add(r.c0, t0, t1);
}
// complex squaring: 2 Fp6 mults
template <class F2>
B3_FN_NOINLINE void fp12_sqr(fp12_t<F2>& r, const fp12_t<F2>& a) {
    fp6_t<F2> ab, s, t;
    fp6_mul(ab, a.c0, a.c1);
    fp6_add(s, a.c0, a.c1);
    fp6_mul_v(t, a.c1);
    fp6_add(t, t, a.c0);
    fp6_mul(s, s, t);                      // (a0+a1)(a0+v a1) = a0^2 + v a1^2 + (1+v) a0 a1
    fp6_sub(s, s, ab);
    fp6_mul_v(t, ab);
    fp6_sub(r.c0, s, t);
    fp6_add(r.c1, ab, ab);
}
// conj = p^6 Frobenius: w -> -w
template <class F2>
B3_FN void fp12_conj(fp12_t<F2>& r, const fp12_t<F2>& a) { r.c0 = a.c0; fp6_neg(r.c1, a.c1); }
template <class F2>
B3_FN_NOINLINE void fp12_inv(fp12_t<F2>& r, const fp12_t<F2>& a) {
    fp6_t<F2> t0, t1;
    fp6_sqr(t0, a.c0);
    fp6_sqr(t1, a.c1);
    fp6_mul_v(t1, t1);
    fp6_sub(t0, t0, t1);
    fp6_inv(t0, t0);
    fp6_mul(r.c0, a.c0, t0);
    fp6_mul(t1, a.c1, t0);
    fp6_neg(r.c1, t1);
}
// multiply by a sparse line  l0 + l3 w^3 + l5 w^5  =  (l0,0,0) + (0,l3,l5) w
template <class F2>
B3_FN_NOINLINE void fp12_mul_by_line(fp12_t<F2>& f, const F2& l0, const F2& l3, const F2& l5) {
    fp6_t<F2> t0, t1, s;
    fp6_mul_fp2(t0, f.c0, l0);                       // f0 * L0
    fp6_mul_by_12(t1, f.c1, l3, l5);                 // f1 * L1
    fp6_add(s, f.c0, f.c1);
    fp6_t<F2> L;
    L.c0 = l0; L.c1 = l3; L.c2 = l5;
    fp6_mul(s, s, L);                                // (f0+f1)(L0+L1)
    fp6_sub(s, s, t0);
    fp6_sub(f.c1, s, t1);
    fp6_mul_v(t1, t1);
    fp6_add(f.c0, t0, t1);
}

// Sparse-line product by dot products: r = f * (l0 + l3 w^3 + l5 w^5), r must not alias f.
// In the w-power basis f = sum f_k w^k (w^6 = xi):
//   r_k = l0 f_k + L3 f_{k-3 mod 6} + L5 f_{k-5 mod 6},   L3 = l3 (k >= 3) or xi l3,   L5 = l5 (k = 5) or xi l5,
// and every Fp coordinate of r_k is ONE six-term dot product with a single Montgomery reduction (fp_dot6):
//   re = sum X0 F0 + (-X1) F1,   im = sum X0 F1 + X1 F0     over the three (X, F) pairs.
// 12 x 1020 multiply-accumulates and no Fp2 additions, against 14 Fp2 products plus ~40 Fp2 additions for the
// Karatsuba form (fp12_mul_by_line).
struct line_ops {                // operands of one line, prepared once
    fp c0[5], c1[5], n1[5];      // X.c0, X.c1, -X.c1 for X = l0, l3, xi l3, l5, xi l5
};
B3_FN_NOINLINE void line_ops_make(line_ops& o, const fp2& l0, const fp2& l3, const fp2& l5) {
    fp2 x3, x5;
    fp2_mul_xi(x3, l3);
    fp2_mul_xi(x5, l5);
    const fp2* src[5] = {&l0, &l3, &x3, &l5, &x5};
    for (int i = 0; i < 5; i++) {
        o.c0[i] = src[i]->c0;
        o.c1[i] = src[i]->c1;
        fp_neg(o.n1[i], src[i]->c1);
    }
}
B3_FN_NOINLINE void fp12_mul_by_line_dot(fp12& r, const fp12& f, const line_ops& o) {
    const fp2* fc = reinterpret_cast<const fp2*>(&f);
    fp2* rc = reinterpret_cast<fp2*>(&r);
#pragma unroll 1
    for (int k = 0; k < 6; k++) {
        const int j3 = k >= 3 ? k - 3 : k + 3, j5 = k == 5 ? 0 : k + 1;
        const int x3 = k >= 3 ? 1 : 2, x5 = k == 5 ? 3 : 4;                   // index into line_ops
        // memory slot of w-power m in an fp12: even m -> m/2, odd m -> 3 + m/2
        const fp2& F0 = fc[(k & 1) ? 3 + (k >> 1) : (k >> 1)];
        const fp2& F3 = fc[(j3 & 1) ? 3 + (j3 >> 1) : (j3 >> 1)];
        const fp2& F5 = fc[(j5 & 1) ? 3 + (j5 >> 1) : (j5 >> 1)];
        fp2& R = rc[(k & 1) ? 3 + (k >> 1) : (k >> 1)];
        fp_dot6_args q;
        q.a[0] = &F0.c0; q.b[0] = &o.c0[0];  q.a[1] = &F0.c1; q.b[1] = &o.n1[0];
        q.a[2] = &F3.c0; q.b[2] = &o.c0[x3]; q.a[3] = &F3.c1; q.b[3] = &o.n1[x3];
        q.a[4] = &F5.c0; q.b[4] = &o.c0[x5]; q.a[5] = &F5.c1; q.b[5] = &o.n1[x5];
        fp_dot6(R.c0, q);
        q.a[0] = &F0.c1; q.b[0] = &o.c0[0];  q.a[1] = &F0.c0; q.b[1] = &o.c1[0];
        q.a[2] = &F3.c1; q.b[2] = &o.c0[x3]; q.a[3] = &F3.c0; q.b[3] = &o.c1[x3];
        q.a[4] = &F5.c1; q.b[4] = &o.c0[x5]; q.a[5] = &F5.c0; q.b[5] = &o.c1[x5];
        fp_dot6(R.c1, q);
    }
}

// p-power Frobenius: f_k -> conj(f_k) * GAMMA1[k]
template <class F2>
B3_FN F2& fp12_coef(fp12_t<F2>& a, int k) {
    return (k & 1) ? ((k == 1) ? a.c1.c0 : (k == 3) ? a.c1.c1 : a.c1.c2)
                   : ((k == 0) ? a.c0.c0 : (k == 2) ? a.c0.c1 : a.c0.c2);
}
template <class F2>
B3_FN const F2& fp12_coef(const fp12_t<F2>& a, int k) {
    return (k & 1) ? ((k == 1) ? a.c1.c0 : (k == 3) ? a.c1.c1 : a.c1.c2)
                   : ((k == 0) ? a.c0.c0 : (k == 2) ? a.c0.c1 : a.c0.c2);
}
template <class F2>
B3_FN_NOINLINE void fp12_frob(fp12_t<F2>& r, const fp12_t<F2>& a) {
    for (int k = 0; k < 6; k++) {
        F2 t;
        fp2_conj(t, fp12_coef(a, k));
        if (k == 0) fp12_coef(r, 0) = t;
        else { F2 g; f2_const(g, FROB_GAMMA1[k]); fp2_mul(fp12_coef(r, k), t, g); }
    }
}
template <class F2>
B3_FN_NOINLINE void fp12_frob2(fp12_t<F2>& r, const fp12_t<F2>& a) {
    fp12_coef(r, 0) = fp12_coef(a, 0);
    for (int k = 1; k < 6; k++) fp2_mul_fp(fp12_coef(r, k), fp12_coef(a, k), FROB_GAMMA2[k]);
}
template <class F2>
B3_FN_NOINLINE void fp12_frob3(fp12_t<F2>& r, const fp12_t<F2>& a) {
    for (int k = 0; k < 6; k++) {
        F2 t;
        fp2_conj(t, fp12_coef(a, k));
        if (k == 0) fp12_coef(r, 0) = t;
        else { F2 g; f2_const(g, FROB_GAMMA3[k]); fp2_mul(fp12_coef(r, k), t, g); }
    }
}

// Granger-Scott squaring for elements of the cyclotomic subgroup (after the easy part of fexp).
// Uses the Fp4 = Fp2[s]/(s^2 - xi) sub-structure with s = w^3: pairs (f0,f3), (f1,f4), (f2,f5).
template <class F2>
B3_FN_NOINLINE void fp4_sqr_parts(F2& r0, F2& r1, const F2& a, const F2& b) {
    // (a + b s)^2 = (a^2 + xi b^2) + (2ab) s
    F2 t0, t1, t2;
    fp2_sqr(t0, a);
    fp2_sqr(t1, b);
    fp2_add(t2, a, b);
    fp2_sqr(t2, t2);
    fp2_sub(t2, t2, t0);
    fp2_sub(r1, t2, t1);
    fp2_mul_xi(t1, t1);
    fp2_add(r0, t0, t1);
}
template <class F2>
B3_FN_NOINLINE void fp12_cyclo_sqr(fp12_t<F2>& r, const fp12_t<F2>& a) {
    // basis: a = g0 + g1 y + g2 y^2 with y = w (y^3 = s = w^3), g0 = (f0, f3), g1 = (f1, f4), g2 = (f2, f5) in Fp4.
    // Granger-Scott: with A = g0^2, B = g2^2 * s, C = g1^2 :
    //   r.g0 = 3A - 2 conj(g0);  r.g1 = 3B + 2 conj(g1);  r.g2 = 3C - 2 conj(g2)     (conj: s -> -s)
    F2 A0, A1, B0, B1, C0, C1, t;
    const F2 &f0 = fp12_coef(a, 0), &f1 = fp12_coef(a, 1), &f2 = fp12_coef(a, 2),
              &f3 = fp12_coef(a, 3), &f4 = fp12_coef(a, 4), &f5 = fp12_coef(a, 5);
    fp4_sqr_parts(A0, A1, f0, f3);
    fp4_sqr_parts(C0, C1, f1, f4);
    fp4_sqr_parts(B0, B1, f2, f5);
    // B * s : (b0 + b1 s) s = xi b1 + b0 s
    fp2_mul_xi(t, B1);
    B1 = B0;
    B0 = t;
    F2 o0, o1, o2, o3, o4, o5;
    // g0' = 3A - 2 conj(g0) = (3A0 - 2 f0) + (3A1 + 2 f3) s
    fp2_sub(t, A0, f0); fp2_dbl(t, t); fp2_add(o0, t, A0);
    fp2_add(t, A1, f3); fp2_dbl(t, t); fp2_add(o3, t, A1);
    // g1' = 3B + 2 conj(g1) = (3B0 + 2 f1) + (3B1 - 2 f4) s
    fp2_add(t, B0, f1); fp2_dbl(t, t); fp2_add(o1, t, B0);
    fp2_sub(t, B1, f4); fp2_dbl(t, t); fp2_add(o4, t, B1);
    // g2' = 3C - 2 conj(g2) = (3C0 - 2 f2) + (3C1 + 2 f5) s
    fp2_sub(t, C0, f2); fp2_dbl(t, t); fp2_add(o2, t, C0);
    fp2_add(t, C1, f5); fp2_dbl(t, t); fp2_add(o5, t, C1);
    fp12_coef(r, 0) = o0; fp12_coef(r, 1) = o1; fp12_coef(r, 2) = o2;
    fp12_coef(r, 3) = o3; fp12_coef(r, 4) = o4; fp12_coef(r, 5) = o5;
}

// Wire format of the reference (A/fp12.rs:859-913): 12 x 48-byte big-endian canonical coefficients in the
// order w^0, w^3, w^1, w^4, w^2, w^5, each (re, im).
B3_FN_NOINLINE void fp12_to_wire(uint8_t* out, const fp12& a) {
    const int order[6] = {0, 3, 1, 4, 2, 5};
    for (int k = 0; k < 6; k++) {
        const fp2& c = fp12_coef(a, order[k]);
        fp t;
        fp_from_mont(t, c.c0);
        fp_raw_to_be(out + 96 * k, t);
        fp_from_mont(t, c.c1);
        fp_raw_to_be(out + 96 * k + 48, t);
    }
}
