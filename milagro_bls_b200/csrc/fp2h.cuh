// Fp2 on LANE PAIRS: lanes (2k, 2k+1) of a warp hold one Fp2 value, the even lane its real part c0, the odd lane its
// imaginary part c1.  Every routine below is executed by both lanes of the pair in lock step (uniform control flow
// inside a pair; different pairs of a warp may diverge -- the shuffles name only the pair in their mask).
//
// This doubles the thread count of every G2 / Fp2 chain of the path (subgroup checks, [c]sig, cofactor clearing,
// Miller point chains), whose outer parallelism -- one item per signature set -- is too small to fill 148 SMs.
//   add/sub/neg/dbl/half/mul_fp : each lane on its own half, no communication
//   mul : one exchange, then each lane one dual product with a single reduction (fp_mul2):
//           even: a0 b0 + (-a1) b1        odd: a0 b1 + a1 b0
//   sqr : one exchange, then each lane ONE Fp product:  even: (a0 + a1)(a0 - a1)   odd: (2 a0) a1
// The overloads use the same names as the single-thread fp2 routines (tower.cuh), so the point formulas of
// curve.cuh / pairing.cuh, written as templates over the field type, work on either representation.
#pragma once
#include "curve.cuh"

#if !defined(B3_HOSTSIM)
struct fp2h {
    fp v;
};

__device__ __forceinline__ unsigned pair_mask() { return 3u << (threadIdx.x & 30u); }
__device__ __forceinline__ bool pair_odd() { return (threadIdx.x & 1u) != 0; }
__device__ __forceinline__ void pair_xchg(fp& r, const fp& a) {
    const unsigned m = pair_mask();
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = __shfl_xor_sync(m, a.l[i], 1);
}
__device__ __forceinline__ bool pair_and(bool x) {
    const int mine = x ? 1 : 0;
    const int other = __shfl_xor_sync(pair_mask(), mine, 1);      // unconditional: both lanes must execute the shuffle
    return (mine & other) != 0;
}

// this lane's half of a full Fp2 value in memory / of a constant
__device__ __forceinline__ void fp2h_load(fp2h& r, const fp2& a) { r.v = (&a.c0)[pair_odd() ? 1 : 0]; }
__device__ __forceinline__ void fp2h_store(fp2& a, const fp2h& r) { (&a.c0)[pair_odd() ? 1 : 0] = r.v; }
__device__ __forceinline__ void f2_const(fp2h& r, const fp2& c) { fp2h_load(r, c); }

B3_FN void fp2_add(fp2h& r, const fp2h& a, const fp2h& b) { fp_add(r.v, a.v, b.v); }
B3_FN void fp2_sub(fp2h& r, const fp2h& a, const fp2h& b) { fp_sub(r.v, a.v, b.v); }
B3_FN void fp2_neg(fp2h& r, const fp2h& a) { fp_neg(r.v, a.v); }
B3_FN void fp2_dbl(fp2h& r, const fp2h& a) { fp_dbl(r.v, a.v); }
B3_FN void fp2_half(fp2h& r, const fp2h& a) { fp_half(r.v, a.v); }
B3_FN void fp2_mul3(fp2h& r, const fp2h& a) { fp t; fp_dbl(t, a.v); fp_add(r.v, t, a.v); }
B3_FN void fp2_conj(fp2h& r, const fp2h& a) {
    fp t;
    fp_neg(t, a.v);
    fp_select(r.v, pair_odd(), t, a.v);
}
B3_FN bool fp2_is_zero(const fp2h& a) { return pair_and(fp_is_zero(a.v)); }
B3_FN bool fp2_eq(const fp2h& a, const fp2h& b) { return pair_and(fp_eq(a.v, b.v)); }
B3_FN void fp2_select(fp2h& r, bool c, const fp2h& a, const fp2h& b) { fp_select(r.v, c, a.v, b.v); }
B3_FN void fp2_zero(fp2h& r) { r.v = FP_NIL; }
B3_FN void fp2_one(fp2h& r) { fp_select(r.v, pair_odd(), FP_NIL, FP_ONE); }
B3_FN_NOINLINE fp2h fp2h_mul_v(fp2h a, fp2h b) {
    fp ao, bo, nao, x1, x2;
    pair_xchg(ao, a.v);
    pair_xchg(bo, b.v);
    fp_neg_nr(nao, ao);
    const bool odd = pair_odd();
    fp_select(x1, odd, ao, a.v);          // even: a0      odd: a0
    fp_select(x2, odd, a.v, nao);         // even: -a1     odd: a1
    fp2h r;
    fp_mul2_inl(r.v, x1, b.v, x2, bo);    // even: a0 b0 - a1 b1     odd: a0 b1 + a1 b0
    return r;
}
B3_FN void fp2_mul(fp2h& r, const fp2h& a, const fp2h& b) { r = fp2h_mul_v(a, b); }
B3_FN_NOINLINE fp2h fp2h_sqr_v(fp2h a) {
    fp ao, x, y, d;
    pair_xchg(ao, a.v);
    const bool odd = pair_odd();
    fp_select(x, odd, ao, a.v);
    fp_add_nr(x, x, ao);                  // even: a0 + a1   odd: 2 a0     (< 4p: the first operand of the product)
    fp_sub(d, a.v, ao);
    fp_select(y, odd, a.v, d);            // even: a0 - a1   odd: a1
    fp2h r;
    fp_mul_inl(r.v, x, y);
    return r;
}
B3_FN void fp2_sqr(fp2h& r, const fp2h& a) { r = fp2h_sqr_v(a); }
B3_FN void fp2_mul_fp(fp2h& r, const fp2h& a, const fp& s) { fp_mul(r.v, a.v, s); }
// * xi = (1 + i): (a0 - a1) + (a0 + a1) i
B3_FN void fp2_mul_xi(fp2h& r, const fp2h& a) {
    fp ao, s, d;
    pair_xchg(ao, a.v);
    fp_add(s, a.v, ao);
    fp_sub(d, a.v, ao);
    fp_select(r.v, pair_odd(), s, d);
}
// 1/a = conj(a) / (a0^2 + a1^2); 0 -> 0.  Both lanes run the (identical) Fp inversion.
B3_FN_NOINLINE void fp2_inv(fp2h& r, const fp2h& a) {
    fp n, no, t;
    fp_sqr(n, a.v);
    pair_xchg(no, n);
    fp_add(n, n, no);
    fp_inv(n, n);
    fp_mul(t, a.v, n);
    fp_neg(no, t);
    fp_select(r.v, pair_odd(), no, t);
}

B3_FN void f_add(fp2h& r, const fp2h& a, const fp2h& b) { fp2_add(r, a, b); }
B3_FN void f_sub(fp2h& r, const fp2h& a, const fp2h& b) { fp2_sub(r, a, b); }
B3_FN void f_mul(fp2h& r, const fp2h& a, const fp2h& b) { fp2_mul(r, a, b); }
B3_FN void f_sqr(fp2h& r, const fp2h& a) { fp2_sqr(r, a); }
B3_FN void f_dbl(fp2h& r, const fp2h& a) { fp2_dbl(r, a); }
B3_FN void f_neg(fp2h& r, const fp2h& a) { fp2_neg(r, a); }
B3_FN void f_inv(fp2h& r, const fp2h& a) { fp2_inv(r, a); }
B3_FN bool f_is_zero(const fp2h& a) { return fp2_is_zero(a); }
B3_FN bool f_eq(const fp2h& a, const fp2h& b) { return fp2_eq(a, b); }
B3_FN void f_select(fp2h& r, bool c, const fp2h& a, const fp2h& b) { fp2_select(r, c, a, b); }
B3_FN void f_one(fp2h& r) { fp2_one(r); }
B3_FN void f_zero(fp2h& r) { fp2_zero(r); }
B3_FN void f_mul_b(fp2h& r, const fp2h& a) { fp2h t; fp2_dbl(t, a); fp2_dbl(t, t); fp2_mul_xi(r, t); }

typedef jac<fp2h> g2h_jac;
typedef aff<fp2h> g2h_aff;

// full <-> lane-pair conversions of points that live in memory
__device__ __forceinline__ void g2h_load(g2h_jac& r, const g2_jac& a) { fp2h_load(r.x, a.x); fp2h_load(r.y, a.y); fp2h_load(r.z, a.z); }
__device__ __forceinline__ void g2h_store(g2_jac& a, const g2h_jac& r) { fp2h_store(a.x, r.x); fp2h_store(a.y, r.y); fp2h_store(a.z, r.z); }
__device__ __forceinline__ void g2h_load(g2h_aff& r, const g2_aff& a) { fp2h_load(r.x, a.x); fp2h_load(r.y, a.y); r.inf = a.inf; }
#endif
