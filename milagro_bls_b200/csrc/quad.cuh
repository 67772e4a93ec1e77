// REPLICATED representations: twice the lanes per item for the latency-bound point chains of a single call.
//
// A verification call of 8192 sets gives the chain kernels one item per set: with one thread (G1) or one lane pair (G2) per
// item that is 256 / 512 warps for 592 SM sub-partitions -- at most one warp each, where a dependent chain of Montgomery
// products reaches 63 % of the multiplier's rate (profiles/microbench/r1s_fpbench.txt) and most of the machine idles.
// Here every value of a chain is held TWICE -- fpd: an Fp value in both lanes of a lane pair; fp2q: a lane-pair Fp2 value
// (fp2h.cuh) in both pairs of a lane quad -- and the point formulas name their independent products in pairs
// (curve.cuh: f_mul_par / f_sqr_par / f_mulsqr_par): each half of the group computes ONE product of the pair, then the
// halves swap results (12 shuffles).  Additions, selections and the unpaired products run redundantly on both halves, so
// control flow stays uniform inside the group and nothing else has to be communicated.
//   G1/G2 doubling (2M + 5S)    : 4 rounds instead of 7 products        G2 mixed addition (7M + 4S): 6 instead of 11
//   Miller doubling step (3M+6S): 5 rounds instead of 9                 Miller addition step (16M + 2S): 9 instead of 18
// A squaring paired with a multiplication runs as a multiplication (both halves of a warp execute one instruction stream).
// The chain kernels are templates over the lane layouts at the end of this file.  Their replicated instantiations
// (lanes_pair for G1, lanes_quad for G2) do ~25 % more multiply-accumulates than the plain ones (lanes_thread, lanes_pair),
// so they run only when a call cannot fill the GPU by itself (capi.cu: latency_mode).
#pragma once
#include "fp2h.cuh"

#if !defined(B3_HOSTSIM)
// ---------------------------------------------------------------------------------------------- fpd: Fp on a lane pair
struct fpd {
    fp v;
};
B3_FN void f_add(fpd& r, const fpd& a, const fpd& b) { fp_add(r.v, a.v, b.v); }
B3_FN void f_sub(fpd& r, const fpd& a, const fpd& b) { fp_sub(r.v, a.v, b.v); }
B3_FN void f_mul(fpd& r, const fpd& a, const fpd& b) { fp_mul(r.v, a.v, b.v); }
B3_FN void f_sqr(fpd& r, const fpd& a) { fp_sqr(r.v, a.v); }
B3_FN void f_dbl(fpd& r, const fpd& a) { fp_dbl(r.v, a.v); }
B3_FN void f_neg(fpd& r, const fpd& a) { fp_neg(r.v, a.v); }
B3_FN bool f_is_zero(const fpd& a) { return fp_is_zero(a.v); }
B3_FN bool f_eq(const fpd& a, const fpd& b) { return fp_eq(a.v, b.v); }
B3_FN void f_select(fpd& r, bool c, const fpd& a, const fpd& b) { fp_select(r.v, c, a.v, b.v); }
B3_FN void f_one(fpd& r) { r.v = FP_ONE; }
B3_FN void f_zero(fpd& r) { r.v = FP_NIL; }
B3_FN void f_mul_b(fpd& r, const fpd& a) { fp t; fp_dbl(t, a.v); fp_dbl(r.v, t); }
B3_FN const fp& fp_of(const fpd& a) { return a.v; }      // every lane holds the whole value
// the odd lane takes the second product of the pair
B3_FN void f_mul_par(fpd& r1, const fpd& a1, const fpd& b1, fpd& r2, const fpd& a2, const fpd& b2) {
    const bool odd = pair_odd();
    fp x, y, o;
    fp_select(x, odd, a2.v, a1.v);
    fp_select(y, odd, b2.v, b1.v);
    const fp p = fp_mul_v(x, y);
    pair_xchg(o, p);
    fp_select(r1.v, odd, o, p);
    fp_select(r2.v, odd, p, o);
}
B3_FN void f_sqr_par(fpd& r1, const fpd& a1, fpd& r2, const fpd& a2) {
    const bool odd = pair_odd();
    fp x, o;
    fp_select(x, odd, a2.v, a1.v);
    const fp p = fp_sqr_v(x);
    pair_xchg(o, p);
    fp_select(r1.v, odd, o, p);
    fp_select(r2.v, odd, p, o);
}
B3_FN void f_mulsqr_par(fpd& r1, const fpd& a1, const fpd& b1, fpd& r2, const fpd& a2) {
    const bool odd = pair_odd();
    fp x, y, o;
    fp_select(x, odd, a2.v, a1.v);
    fp_select(y, odd, a2.v, b1.v);
    const fp p = fp_mul_v(x, y);
    pair_xchg(o, p);
    fp_select(r1.v, odd, o, p);
    fp_select(r2.v, odd, p, o);
}

// ---------------------------------------------------------------------------------------------- fp2q: Fp2 on a lane quad
// lane l of the quad: half (l & 1) of the Fp2 value as in fp2h, in pair (l >> 1) & 1.  Every fp2h routine applies unchanged
// (each pair runs it on its own copy); only the paired products differ.
struct fp2q : fp2h {};
__device__ __forceinline__ unsigned quad_mask() { return 0xfu << (threadIdx.x & 28u); }
__device__ __forceinline__ bool quad_hi() { return (threadIdx.x & 2u) != 0; }
__device__ __forceinline__ void quad_xchg(fp& r, const fp& a) {
    const unsigned m = quad_mask();
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = __shfl_xor_sync(m, a.l[i], 2);
}
B3_FN void f2_const(fp2q& r, const fp2& c) { fp2h_load(r, c); }
B3_FN void f_mul_par(fp2q& r1, const fp2q& a1, const fp2q& b1, fp2q& r2, const fp2q& a2, const fp2q& b2) {
    const bool hi = quad_hi();
    fp2h x, y;
    fp o;
    fp_select(x.v, hi, a2.v, a1.v);
    fp_select(y.v, hi, b2.v, b1.v);
    const fp2h p = fp2h_mul_v(x, y);
    quad_xchg(o, p.v);
    fp_select(r1.v, hi, o, p.v);
    fp_select(r2.v, hi, p.v, o);
}
B3_FN void f_sqr_par(fp2q& r1, const fp2q& a1, fp2q& r2, const fp2q& a2) {
    const bool hi = quad_hi();
    fp2h x;
    fp o;
    fp_select(x.v, hi, a2.v, a1.v);
    const fp2h p = fp2h_sqr_v(x);
    quad_xchg(o, p.v);
    fp_select(r1.v, hi, o, p.v);
    fp_select(r2.v, hi, p.v, o);
}
B3_FN void f_mulsqr_par(fp2q& r1, const fp2q& a1, const fp2q& b1, fp2q& r2, const fp2q& a2) {
    const bool hi = quad_hi();
    fp2h x, y;
    fp o;
    fp_select(x.v, hi, a2.v, a1.v);
    fp_select(y.v, hi, a2.v, b1.v);
    const fp2h p = fp2h_mul_v(x, y);
    quad_xchg(o, p.v);
    fp_select(r1.v, hi, o, p.v);
    fp_select(r2.v, hi, p.v, o);
}
// ---------------------------------------------------------------------------------------------- lane layouts
// The chain kernels (kernels.cuh) are templates over a lane layout L: item i runs on the 1 << L::shift lanes from
// i << L::shift, holding its G1 values as L::g1 and its G2 values as L::g2.  L::leader() is the one lane of the group that
// writes a single-writer result; L::load / L::store convert between a full point in memory and the group's values.
//   lanes_thread: one thread per item (G1 in fp)
//   lanes_pair  : G1 replicated in fpd, G2 split over the pair in fp2h (fp2h.cuh)
//   lanes_quad  : G2 replicated in fp2q
struct lanes_thread {
    typedef fp g1;
    static constexpr unsigned shift = 0;
    static __device__ __forceinline__ bool leader() { return true; }
    static __device__ __forceinline__ void load(g1_jac& r, const g1_jac& a) { r = a; }
    static __device__ __forceinline__ void store(g1_jac& a, const g1_jac& r) { a = r; }
};
struct lanes_pair {
    typedef fpd g1;
    typedef fp2h g2;
    static constexpr unsigned shift = 1;
    static __device__ __forceinline__ bool leader() { return !pair_odd(); }
    static __device__ __forceinline__ void load(jac<fpd>& r, const g1_jac& a) { r.x.v = a.x; r.y.v = a.y; r.z.v = a.z; }
    static __device__ __forceinline__ void store(g1_jac& a, const jac<fpd>& r) { a.x = r.x.v; a.y = r.y.v; a.z = r.z.v; }
    static __device__ __forceinline__ void load(g2h_jac& r, const g2_jac& a) { g2h_load(r, a); }
    static __device__ __forceinline__ void load(g2h_aff& r, const g2_aff& a) { g2h_load(r, a); }
    // the coefficients (u0, l3, u5) of a Miller line at o: each lane stores its half of all three
    static __device__ __forceinline__ void store_line(fp2* o, const fp2h& u0, const fp2h& l3, const fp2h& u5) {
        fp2h_store(o[0], u0); fp2h_store(o[1], l3); fp2h_store(o[2], u5);
    }
};
struct lanes_quad {
    typedef fp2q g2;
    static constexpr unsigned shift = 2;
    static __device__ __forceinline__ bool leader() { return (threadIdx.x & 3u) == 0; }
    static __device__ __forceinline__ void load(jac<fp2q>& r, const g2_jac& a) { fp2h_load(r.x, a.x); fp2h_load(r.y, a.y); fp2h_load(r.z, a.z); }
    static __device__ __forceinline__ void load(aff<fp2q>& r, const g2_aff& a) { fp2h_load(r.x, a.x); fp2h_load(r.y, a.y); r.inf = a.inf; }
    // the low pair stores u0 and l3, the high pair u5
    static __device__ __forceinline__ void store_line(fp2* o, const fp2q& u0, const fp2q& l3, const fp2q& u5) {
        if (quad_hi()) fp2h_store(o[2], u5);
        else { fp2h_store(o[0], u0); fp2h_store(o[1], l3); }
    }
};
#endif
