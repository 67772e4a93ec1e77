// Optimal-ate Miller loop and final exponentiation for BLS12-381.
//
// Replaces the reference's per-bit-accumulator multi-pairing
//   /root/reference/incubator-milagro-crypto-rust/src/pair.rs:35-133 (linedbl/lineadd),
//   156-238 (initmp/another/miller), 409-541 (fexp, BLS branch 485-539).
// Only the value AFTER the final exponentiation is comparable with the reference (SURVEY.md B.5): line
// functions here are scaled by Fp2 factors and the loop runs over the plain binary expansion of |x|
// instead of the reference's (3n - n) signed form; both differences vanish in
// GT = m^(3 (p^12 - 1) / r).
#pragma once
#include "curve.cuh"

// ---- split Miller loop (multi-pairing with per-step accumulators, the shape of A/pair.rs:156-238) -----------------
// The point chain T -> 2T (-> T + Q) of a pair depends only on Q, and the lines it produces are independent of the
// accumulator f.  So the loop is split in three data-parallel pieces (kernels.cuh):
//   1. per pair: run the point chain and emit the B3_MILLER_SLOTS lines WITHOUT their P-dependent factors;
//   2. per (slot, pair): scale the line by (xP, -yP) and multiply it into the slot's accumulator  A_s = prod_pairs l_s
//      -- every (slot, pair) is independent, and no per-pair Fp12 squarings are needed;
//   3. once: f = 1; for it = 0..62: f = f^2 * A_it [* A_(63 + k) on the 5 addition steps]; conj.
// Slot it (0..62) holds the doubling line of loop index i = 62 - it; slots 63..67 hold the addition lines in loop order.
#define B3_MILLER_DBL_SLOTS 63
#define B3_MILLER_SLOTS 68
// Unscaled doubling step.  Full line: l0 = u0 * (-yP),  l3,  l5 = u5 * xP   with u0 = xi (2YZ), u5 = 3 X^2.
template <class F2>
struct miller_pt_t {
    F2 x, y, z;
};
template <class F2>
B3_FN_NOINLINE void miller_dbl_step_u(miller_pt_t<F2>& t, F2& u0, F2& l3, F2& u5) {
    F2 a, b, c, e, f, g, h, j, e2, u, g2, x3, z3;
    f_sqr_par(b, t.y, c, t.z);      // B = Y^2, C = Z^2
    fp2_add(h, t.y, t.z);
    f_sqr_par(h, h, j, t.x);        // (Y + Z)^2, J = X^2
    fp2_mul3(u, c);
    f_mul_b(e, u);                  // E = 3 b' C
    fp2_mul3(f, e);                 // F = 3E
    fp2_add(g, b, f);
    fp2_half(g, g);                 // G = (B+F)/2
    fp2_add(u, b, c);
    fp2_sub(h, h, u);               // H = 2YZ
    f_sqr_par(e2, e, g2, g);        // E^2, G^2
    f_mul_par(a, t.x, t.y, z3, b, h);   // XY, Z3 = B H
    fp2_half(a, a);                 // A = XY/2
    fp2_sub(l3, e, b);
    fp2_mul3(u5, j);
    fp2_mul_xi(u0, h);
    fp2_sub(u, b, f);
    f_mul(x3, a, u);                // X3 = A (B - F)
    t.x = x3;
    fp2_mul3(u, e2);
    fp2_sub(t.y, g2, u);            // Y3 = G^2 - 3 E^2
    t.z = z3;
}
// Unscaled addition step T <- T + Q with Q = (X2 : Y2 : Z2) homogeneous projective (x2 = X2/Z2, y2 = Y2/Z2), so that
// hash_to_curve outputs never have to be normalised.  It is the mixed step (A/pair.rs:88-133) with theta, lambda and
// the new point scaled by powers of Z2 -- Fp2 factors, which vanish in the final exponentiation.  Signs are arranged
// so that the same factors (-yP, xP) apply as for a doubling line:
//   l0 = u0 * (-yP), l3, l5 = u5 * xP   with u0 = -xi lambda Z2, l3 = theta X2 - lambda Y2, u5 = -theta Z2,
//   theta = Y1 Z2 - Y2 Z1,  lambda = X1 Z2 - X2 Z1.
template <class F2>
B3_FN_NOINLINE void miller_add_step_u(miller_pt_t<F2>& t, F2& u0, F2& l3, F2& u5, const F2& xq, const F2& yq, const F2& zq) {
    F2 theta, lambda, c, d, e, f, g, h, u, v, xz, yz, zz, x3, z3;
    f_mul_par(xz, t.x, zq, yz, t.y, zq);
    f_mul_par(zz, t.z, zq, u, yq, t.z);
    fp2_sub(theta, yz, u);
    f_mulsqr_par(v, xq, t.z, c, theta);
    fp2_sub(lambda, xz, v);
    f_mulsqr_par(f, zz, c, d, lambda);
    f_mul_par(e, lambda, d, g, xz, d);
    fp2_add(h, e, f);
    fp2_sub(h, h, g);
    fp2_sub(h, h, g);               // H = E + F - 2G
    f_mul_par(l3, theta, xq, u, lambda, yq);
    fp2_sub(l3, l3, u);
    f_mul_par(u, theta, zq, v, lambda, zq);
    fp2_neg(u5, u);
    fp2_mul_xi(v, v);
    fp2_neg(u0, v);
    fp2_sub(u, g, h);
    f_mul_par(x3, lambda, h, v, theta, u);
    f_mul_par(g, e, yz, z3, zz, e);
    t.x = x3;
    fp2_sub(t.y, v, g);
    t.z = z3;
}
// Start of a point chain from a Jacobian Q = (X : Y : Z), x = X/Z^2, y = Y/Z^3: homogeneous (X Z : Y : Z^3)
template <class F2>
B3_FN void miller_start(miller_pt_t<F2>& t, const F2& X, const F2& Y, const F2& Z) {
    F2 z2;
    f_mulsqr_par(t.x, X, Z, z2, Z);
    t.y = Y;
    f_mul(t.z, z2, Z);
}
// G1 member of a pairing in the form the line scaling wants: for P = (X : Y : Z) Jacobian (x = X/Z^2, y = Y/Z^3)
// the line  l0 = u0 (-y), l3, l5 = u5 x  times Z^3 is  u0 (-Y), l3 Z^3, u5 (X Z)  -- no inversion.
struct g1_pp {
    fp xz, ny, z3;
    uint32_t inf;
};
// P in any G1 representation whose lanes each hold the whole value (fp; fpd, quad.cuh)
B3_FN const fp& fp_of(const fp& a) { return a; }
template <class F>
B3_FN void g1_pp_from_jac(g1_pp& r, const jac<F>& p) {
    F xz, z2, z3;
    f_mulsqr_par(xz, p.x, p.z, z2, p.z);
    f_mul(z3, z2, p.z);
    r.xz = fp_of(xz);
    fp_neg(r.ny, fp_of(p.y));
    r.z3 = fp_of(z3);
    r.inf = pt_is_inf(p) ? 1u : 0u;
}

// dense Fp12 value of a line  l0 + l3 w^3 + l5 w^5
template <class F2>
B3_FN void fp12_from_line(fp12_t<F2>& f, const F2& l0, const F2& l3, const F2& l5) {
    f.c0.c0 = l0; fp2_zero(f.c0.c1); fp2_zero(f.c0.c2);
    fp2_zero(f.c1.c0); f.c1.c1 = l3; f.c1.c2 = l5;
}

// f^|x| for f in the cyclotomic subgroup (63 cyclotomic squarings + 5 multiplications)
template <class F2>
B3_FN_NOINLINE void fp12_pow_x_abs(fp12_t<F2>& r, const fp12_t<F2>& a, int shift) {
    const uint64_t x = B3_X_ABS >> shift;
    fp12_t<F2> acc = a;
    int top = 63 - shift;
    for (int i = top - 1; i >= 0; i--) {
        fp12_cyclo_sqr(acc, acc);
        if ((x >> i) & 1) fp12_mul(acc, acc, a);
    }
    r = acc;
}
// f^x (x negative): pow(|x|) then conjugate, as the reference does after every pow (A/pair.rs:490-529)
template <class F2>
B3_FN void fp12_pow_x(fp12_t<F2>& r, const fp12_t<F2>& a) { fp12_pow_x_abs(r, a, 0); fp12_conj(r, r); }
template <class F2>
B3_FN void fp12_pow_x_half(fp12_t<F2>& r, const fp12_t<F2>& a) { fp12_pow_x_abs(r, a, 1); fp12_conj(r, r); }

// Final exponentiation: exactly the exponent 3 (p^12 - 1) / r the reference computes
// (easy part (p^6 - 1)(p^2 + 1), hard part = Ghammam-Fouotsa chain of A/pair.rs:485-539).
template <class F2>
B3_FN_NOINLINE void final_exp(fp12_t<F2>& r, const fp12_t<F2>& m) {
    fp12_t<F2> t, y0, y1, y2, y3, rr;
    fp12_inv(t, m);
    fp12_conj(rr, m);
    fp12_mul(rr, rr, t);                // m^(p^6 - 1)
    fp12_frob2(t, rr);
    fp12_mul(rr, t, rr);                // ^(p^2 + 1)
    // hard part
    fp12_cyclo_sqr(y0, rr);             // y0 = r^2
    fp12_pow_x(y1, y0);                 // y1 = y0^x
    fp12_pow_x_half(y2, y1);            // y2 = y1^(x/2)
    fp12_conj(y3, rr);
    fp12_mul(y1, y1, y3);
    fp12_conj(y1, y1);
    fp12_mul(y1, y1, y2);
    fp12_pow_x(y2, y1);
    fp12_pow_x(y3, y2);
    fp12_conj(y1, y1);
    fp12_mul(y3, y3, y1);
    fp12_conj(y1, y1);
    fp12_frob3(y1, y1);
    fp12_frob2(y2, y2);
    fp12_mul(y1, y1, y2);
    fp12_pow_x(y2, y3);
    fp12_mul(y2, y2, y0);
    fp12_mul(y2, y2, rr);
    fp12_mul(y1, y1, y2);
    fp12_frob(y2, y3);
    fp12_mul(r, y1, y2);
}
