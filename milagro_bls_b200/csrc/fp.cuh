// Fp arithmetic for BLS12-381 on sm_100a: 381-bit Montgomery residues, R = 2^384, 12 x 32-bit limbs.
//
// Replaces (does not port) the reference's FP/Big/DBig layer:
//   /root/reference/incubator-milagro-crypto-rust/src/fp.rs:306-314,390-398 (mul/sqr -> Big::mul + Big::monty)
//   /root/reference/incubator-milagro-crypto-rust/src/big.rs:950-986,1064-1106 (7 x 58-bit limbs, R = 2^406)
// The reference's radix and lazy-reduction bookkeeping are not observable (SURVEY.md B.1).  Here every device value
// is a Montgomery residue in [0, 2p), not necessarily the canonical one: p < 2^381 leaves three spare bits under R, so a
// product of two such values, (ab + mp)/R < 4p^2/R + p < 1.41p, needs no final subtraction, and additions and subtractions
// reduce modulo 2p.  The canonical representative (fp_canon) is formed only where a value is compared, tested for zero,
// has its sign or parity read, or leaves the device: fp_is_zero, fp_eq, fp_from_mont, fp_inv and the wire writers.
//
// The multiplier is a row-wise Montgomery product with two 32-bit-staggered accumulators ("even"/"odd"
// columns) so that every 32x32->64 partial product is one `mad.lo.cc`/`madc.hi.cc` pair on an aligned
// register pair, which ptxas fuses into IMAD.WIDE(.X) carry chains.
//
// The same source also compiles with a plain host C++ compiler (B3_HOSTSIM) where the PTX carry-flag
// primitives are emulated; that build exists ONLY for tests/hostsim (CPU-side debugging of the device
// algorithms) and is never linked into the product library.
#pragma once
#include <stdint.h>

#if defined(B3_HOSTSIM)
#define B3_FN static inline
#define B3_FN_NOINLINE static
#define B3_CONST static const
#else
#define B3_FN __device__ __forceinline__
#define B3_FN_NOINLINE __device__ __noinline__
#define B3_CONST static __device__ __constant__ const
#endif

struct alignas(16) fp {
    uint32_t l[12];
};
struct fp2 {
    fp c0, c1;
};

#include "constants.cuh"

// ------------------------------------------------------------------------------------------------
// carry-flag primitives
// ------------------------------------------------------------------------------------------------
#if defined(B3_HOSTSIM)
static thread_local uint32_t b3_cc = 0;
static inline uint32_t add_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a + b; b3_cc = (uint32_t)(t >> 32); return (uint32_t)t; }
static inline uint32_t addc_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a + b + b3_cc; b3_cc = (uint32_t)(t >> 32); return (uint32_t)t; }
static inline uint32_t addc(uint32_t a, uint32_t b) { return a + b + b3_cc; }
static inline uint32_t sub_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a - b; b3_cc = (uint32_t)(t >> 63); return (uint32_t)t; }
static inline uint32_t subc_cc(uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a - b - b3_cc; b3_cc = (uint32_t)(t >> 63); return (uint32_t)t; }
static inline uint32_t subc(uint32_t a, uint32_t b) { return a - b - b3_cc; }
// (lo,hi) = a*b
static inline void mul_wide(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) { uint64_t t = (uint64_t)a * b; lo = (uint32_t)t; hi = (uint32_t)(t >> 32); }
// (lo,hi) += a*b, carry chain started here
static inline void mad_wide_cc(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) {
    uint64_t t = (uint64_t)a * b;
    uint64_t s = (uint64_t)lo + (uint32_t)t; lo = (uint32_t)s;
    s = (uint64_t)hi + (uint32_t)(t >> 32) + (s >> 32); hi = (uint32_t)s; b3_cc = (uint32_t)(s >> 32);
}
// (lo,hi) += a*b + carry-in, carry out
static inline void madc_wide_cc(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) {
    uint64_t t = (uint64_t)a * b;
    uint64_t s = (uint64_t)lo + (uint32_t)t + b3_cc; lo = (uint32_t)s;
    s = (uint64_t)hi + (uint32_t)(t >> 32) + (s >> 32); hi = (uint32_t)s; b3_cc = (uint32_t)(s >> 32);
}
// (lo,hi) = a*b + (lo_in,hi_in) + carry-in, carry out
static inline void madc_wide_cc_in(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b, uint32_t lo_in, uint32_t hi_in) {
    uint64_t t = (uint64_t)a * b;
    uint64_t s = (uint64_t)lo_in + (uint32_t)t + b3_cc; lo = (uint32_t)s;
    s = (uint64_t)hi_in + (uint32_t)(t >> 32) + (s >> 32); hi = (uint32_t)s; b3_cc = (uint32_t)(s >> 32);
}
// (lo,hi) = a*b + carry-in; the high word cannot overflow; carry flag left unspecified
static inline void madc_wide_last(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) {
    uint64_t t = (uint64_t)a * b + b3_cc; lo = (uint32_t)t; hi = (uint32_t)(t >> 32);
}
#else
B3_FN uint32_t add_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("add.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
B3_FN uint32_t addc_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("addc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
B3_FN uint32_t addc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("addc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
B3_FN uint32_t sub_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("sub.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
B3_FN uint32_t subc_cc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("subc.cc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
B3_FN uint32_t subc(uint32_t a, uint32_t b) { uint32_t r; asm volatile("subc.u32 %0, %1, %2;" : "=r"(r) : "r"(a), "r"(b)); return r; }
B3_FN void mul_wide(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) {
    asm volatile("mul.lo.u32 %0, %2, %3; mul.hi.u32 %1, %2, %3;" : "=r"(lo), "=r"(hi) : "r"(a), "r"(b));
}
B3_FN void mad_wide_cc(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) {
    asm volatile("mad.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(lo), "+r"(hi) : "r"(a), "r"(b));
}
B3_FN void madc_wide_cc(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) {
    asm volatile("madc.lo.cc.u32 %0, %2, %3, %0; madc.hi.cc.u32 %1, %2, %3, %1;" : "+r"(lo), "+r"(hi) : "r"(a), "r"(b));
}
B3_FN void madc_wide_cc_in(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b, uint32_t lo_in, uint32_t hi_in) {
    asm volatile("madc.lo.cc.u32 %0, %2, %3, %4; madc.hi.cc.u32 %1, %2, %3, %5;"
                 : "=r"(lo), "=r"(hi) : "r"(a), "r"(b), "r"(lo_in), "r"(hi_in));
}
B3_FN void madc_wide_last(uint32_t& lo, uint32_t& hi, uint32_t a, uint32_t b) {
    asm volatile("madc.lo.cc.u32 %0, %2, %3, 0; madc.hi.u32 %1, %2, %3, 0;" : "=r"(lo), "=r"(hi) : "r"(a), "r"(b));
}
#endif

// NOTE (nvcc 12.9): an inline helper that owns fp-sized locals whose addresses are passed to __noinline__
// functions gets its stack slots mis-merged when it is inlined more than once into one caller (observed:
// two live temporaries of sswu_g2 sharing one slot, tests/hostsim/dbg_sswu.py).  Rule used throughout: such
// helpers are __noinline__ themselves; only helpers without address-taken locals are force-inlined.
// ------------------------------------------------------------------------------------------------
// basic predicates / moves
// ------------------------------------------------------------------------------------------------
// a == 0 mod p for a in [0, 2p): a is 0 or p
B3_FN bool fp_is_zero(const fp& a) {
    uint32_t z = 0, q = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) { z |= a.l[i]; q |= a.l[i] ^ FP_P.l[i]; }
    return z == 0 || q == 0;
}
// r = c ? a : b
B3_FN void fp_select(fp& r, bool c, const fp& a, const fp& b) {
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = c ? a.l[i] : b.l[i];
}
B3_FN void fp_set(fp& r, const fp& a) {
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = a.l[i];
}

// r = t < m ? t : t - m      (m = p or 2p)
B3_FN void fp_cond_sub(fp& r, const uint32_t* t, const fp& m) {
    uint32_t s[12];
    s[0] = sub_cc(t[0], m.l[0]);
#pragma unroll
    for (int i = 1; i < 12; i++) s[i] = subc_cc(t[i], m.l[i]);
    uint32_t borrow = subc(0, 0);          // 0xffffffff if t < m
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = borrow ? t[i] : s[i];
}
// a in [0, 2p) -> the canonical representative in [0, p)
B3_FN void fp_canon(fp& r, const fp& a) { fp_cond_sub(r, a.l, FP_P); }

B3_FN void fp_add(fp& r, const fp& a, const fp& b) {
    uint32_t t[12];
    t[0] = add_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < 11; i++) t[i] = addc_cc(a.l[i], b.l[i]);
    t[11] = addc(a.l[11], b.l[11]);        // a + b < 4p < 2^384: no carry out
    fp_cond_sub(r, t, FP_2P);
}

B3_FN void fp_sub(fp& r, const fp& a, const fp& b) {
    uint32_t t[12];
    t[0] = sub_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < 12; i++) t[i] = subc_cc(a.l[i], b.l[i]);
    uint32_t m = subc(0, 0);               // all-ones if a < b: a - b + 2p in (0, 2p)
    r.l[0] = add_cc(t[0], FP_2P.l[0] & m);
#pragma unroll
    for (int i = 1; i < 11; i++) r.l[i] = addc_cc(t[i], FP_2P.l[i] & m);
    r.l[11] = addc(t[11], FP_2P.l[11] & m);
}

B3_FN bool fp_eq(const fp& a, const fp& b) {
    fp d;
    fp_sub(d, a, b);
    return fp_is_zero(d);
}

// r = 2p - a, and 0 for a = 0 (so that the result stays below 2p)
B3_FN void fp_neg(fp& r, const fp& a) {
    uint32_t z = 0;
#pragma unroll
    for (int i = 0; i < 12; i++) z |= a.l[i];
    uint32_t t[12];
    t[0] = sub_cc(FP_2P.l[0], a.l[0]);
#pragma unroll
    for (int i = 1; i < 11; i++) t[i] = subc_cc(FP_2P.l[i], a.l[i]);
    t[11] = subc(FP_2P.l[11], a.l[11]);
#pragma unroll
    for (int i = 0; i < 12; i++) r.l[i] = z == 0 ? 0u : t[i];
}

B3_FN void fp_dbl(fp& r, const fp& a) { fp_add(r, a, a); }

// Unreduced forms, for an operand that goes straight into a product and nowhere else (see fp_mul_inl for the bounds):
// r = a + b < 4p, and r = 2p - a in (0, 2p].
B3_FN void fp_add_nr(fp& r, const fp& a, const fp& b) {
    r.l[0] = add_cc(a.l[0], b.l[0]);
#pragma unroll
    for (int i = 1; i < 11; i++) r.l[i] = addc_cc(a.l[i], b.l[i]);
    r.l[11] = addc(a.l[11], b.l[11]);
}
B3_FN void fp_neg_nr(fp& r, const fp& a) {
    r.l[0] = sub_cc(FP_2P.l[0], a.l[0]);
#pragma unroll
    for (int i = 1; i < 11; i++) r.l[i] = subc_cc(FP_2P.l[i], a.l[i]);
    r.l[11] = subc(FP_2P.l[11], a.l[11]);
}

// r = a/2 mod p: (a + p)/2 < 1.5p for odd a, a/2 < p for even a
B3_FN void fp_half(fp& r, const fp& a) {
    uint32_t m = 0u - (a.l[0] & 1u);
    uint32_t t[12];
    t[0] = add_cc(a.l[0], FP_P.l[0] & m);
#pragma unroll
    for (int i = 1; i < 11; i++) t[i] = addc_cc(a.l[i], FP_P.l[i] & m);
    t[11] = addc(a.l[11], FP_P.l[11] & m);  // < 3p < 2^384
#pragma unroll
    for (int i = 0; i < 11; i++) r.l[i] = (t[i] >> 1) | (t[i + 1] << 31);
    r.l[11] = t[11] >> 1;
}

// ------------------------------------------------------------------------------------------------
// Montgomery multiplication  r = a * b / 2^384 mod p, r < 2p      (a, b <= 2p; or a < 4p and b < 2p; or a < p and b any
// 384-bit value).  The running value of the row-wise reduction stays below a + p < 5p < 2^384, so the two 12-limb
// accumulators do not overflow; the result (ab + mp)/2^384 < 8p^2/2^384 + p < 1.82p (or < p + p for the last form) needs
// no final subtraction.
// ------------------------------------------------------------------------------------------------
// acc[0..11] = sum_{j even} x[j] * y * 2^(32 j)            (no carries: products do not overlap)
B3_FN void b3_mul_row(uint32_t* acc, const uint32_t* x, uint32_t y) {
#pragma unroll
    for (int j = 0; j < 12; j += 2) mul_wide(acc[j], acc[j + 1], x[j], y);
}
// acc[0..11] += sum_{j even} x[j] * y * 2^(32 j); carry out left in the flag
B3_FN void b3_mad_row(uint32_t* acc, const uint32_t* x, uint32_t y) {
    mad_wide_cc(acc[0], acc[1], x[0], y);
#pragma unroll
    for (int j = 2; j < 12; j += 2) madc_wide_cc(acc[j], acc[j + 1], x[j], y);
}
// acc = (acc >> 64) + sum_{j even} x[j] * y * 2^(32 j) + carry-in
B3_FN void b3_mad_row_shift(uint32_t* acc, const uint32_t* x, uint32_t y) {
#pragma unroll
    for (int j = 0; j < 10; j += 2) madc_wide_cc_in(acc[j], acc[j + 1], x[j], y, acc[j + 2], acc[j + 3]);
    madc_wide_last(acc[10], acc[11], x[10], y);
}
// one row: (E + 2^32 O) <- ((E + 2^32 O) + a*bi + m*p) / 2^32, roles of E and O swap afterwards
B3_FN void b3_mont_row(uint32_t* even, uint32_t* odd, const uint32_t* a, uint32_t bi, bool first) {
    if (first) {
        b3_mul_row(odd, a + 1, bi);
        b3_mul_row(even, a, bi);
    } else {
        even[0] = add_cc(even[0], odd[1]);
        b3_mad_row_shift(odd, a + 1, bi);
        b3_mad_row(even, a, bi);
        odd[11] = addc(odd[11], 0);
    }
    uint32_t m = even[0] * FP_PINV32;
    b3_mad_row(odd, FP_P.l + 1, m);
    b3_mad_row(even, FP_P.l, m);
    odd[11] = addc(odd[11], 0);
}

B3_FN void fp_mul_inl(fp& r, const fp& a, const fp& b) {
    uint32_t even[12], odd[12], av[12], bv[12];
#pragma unroll
    for (int i = 0; i < 12; i++) { av[i] = a.l[i]; bv[i] = b.l[i]; }
#pragma unroll
    for (int i = 0; i < 12; i += 2) {
        b3_mont_row(even, odd, av, bv[i], i == 0);
        b3_mont_row(odd, even, av, bv[i + 1], false);
    }
    r.l[0] = add_cc(even[0], odd[1]);
#pragma unroll
    for (int i = 1; i < 11; i++) r.l[i] = addc_cc(even[i], odd[i + 1]);
    r.l[11] = addc(even[11], 0);
}

// Dual product with ONE reduction:  r = (a1*b1 + a2*b2) / 2^384 mod p, r < 2p      (a1, a2 <= 2p; b1, b2 < 2p)
// 2 x 144 + 156 multiply-accumulates instead of 2 x 300.  The running value stays below (a1 + a2 + p)(1 + 2^-32) < 5.01p
// < 2^384 and the result below 8p^2/2^384 + p < 1.82p, so the accumulator shapes of fp_mul_inl carry over and there is no
// final subtraction.
B3_FN void b3_mont_row2(uint32_t* even, uint32_t* odd, const uint32_t* a1, uint32_t b1i, const uint32_t* a2, uint32_t b2i, bool first) {
    if (first) {
        b3_mul_row(odd, a1 + 1, b1i);
        b3_mul_row(even, a1, b1i);
    } else {
        even[0] = add_cc(even[0], odd[1]);
        b3_mad_row_shift(odd, a1 + 1, b1i);
        b3_mad_row(even, a1, b1i);
        odd[11] = addc(odd[11], 0);
    }
    b3_mad_row(odd, a2 + 1, b2i);
    b3_mad_row(even, a2, b2i);
    odd[11] = addc(odd[11], 0);
    uint32_t m = even[0] * FP_PINV32;
    b3_mad_row(odd, FP_P.l + 1, m);
    b3_mad_row(even, FP_P.l, m);
    odd[11] = addc(odd[11], 0);
}
B3_FN void fp_mul2_inl(fp& r, const fp& a1, const fp& b1, const fp& a2, const fp& b2) {
    uint32_t even[12], odd[12], a1v[12], b1v[12], a2v[12], b2v[12];
#pragma unroll
    for (int i = 0; i < 12; i++) { a1v[i] = a1.l[i]; b1v[i] = b1.l[i]; a2v[i] = a2.l[i]; b2v[i] = b2.l[i]; }
#pragma unroll
    for (int i = 0; i < 12; i += 2) {
        b3_mont_row2(even, odd, a1v, b1v[i], a2v, b2v[i], i == 0);
        b3_mont_row2(odd, even, a1v, b1v[i + 1], a2v, b2v[i + 1], false);
    }
    r.l[0] = add_cc(even[0], odd[1]);
#pragma unroll
    for (int i = 1; i < 11; i++) r.l[i] = addc_cc(even[i], odd[i + 1]);
    r.l[11] = addc(even[11], 0);
}
// Six-term dot product with ONE reduction:  r = (sum_{t<6} a[t] * b[t]) / 2^384 mod p, r < 2p     (all operands < 2p)
// 6 x 144 + 156 = 1020 multiply-accumulates instead of 6 x 300 plus five additions.  The running value is below
// (sum a[t] + p)(1 + 2^-32): six operands below 2p would reach 13p > 2^384, so the a[t] are made canonical on load and it
// stays below 7p(1 + 2^-32) < 2^384.  The result is below 12p^2/2^384 + p < 2.22p: one conditional subtraction of 2p.
// Operands are read through pointers (they live in local/shared memory: Fp12 accumulators).
struct fp_dot6_args {
    const fp* a[6];
    const fp* b[6];
};
B3_FN_NOINLINE void fp_dot6(fp& r, fp_dot6_args q) {
    uint32_t even[12], odd[12], av[6][12];
#pragma unroll
    for (int t = 0; t < 6; t++) {
#pragma unroll
        for (int i = 0; i < 12; i++) av[t][i] = q.a[t]->l[i];
        fp c;
        fp_cond_sub(c, av[t], FP_P);
#pragma unroll
        for (int i = 0; i < 12; i++) av[t][i] = c.l[i];
    }
#pragma unroll
    for (int i = 0; i < 12; i++) {
        uint32_t* E = (i & 1) ? odd : even;
        uint32_t* O = (i & 1) ? even : odd;
        uint32_t bi = q.b[0]->l[i];
        if (i == 0) {
            b3_mul_row(O, av[0] + 1, bi);
            b3_mul_row(E, av[0], bi);
        } else {
            E[0] = add_cc(E[0], O[1]);
            b3_mad_row_shift(O, av[0] + 1, bi);
            b3_mad_row(E, av[0], bi);
            O[11] = addc(O[11], 0);
        }
#pragma unroll
        for (int t = 1; t < 6; t++) {
            bi = q.b[t]->l[i];
            b3_mad_row(O, av[t] + 1, bi);
            b3_mad_row(E, av[t], bi);
            O[11] = addc(O[11], 0);
        }
        uint32_t m = E[0] * FP_PINV32;
        b3_mad_row(O, FP_P.l + 1, m);
        b3_mad_row(E, FP_P.l, m);
        O[11] = addc(O[11], 0);
    }
    even[0] = add_cc(even[0], odd[1]);
#pragma unroll
    for (int i = 1; i < 11; i++) even[i] = addc_cc(even[i], odd[i + 1]);
    even[11] = addc(even[11], 0);
    fp_cond_sub(r, even, FP_2P);
}

#if !defined(B3_HOSTSIM)
// Register-resident dot product for the group-cooperative Miller accumulation (kernels.cuh, k_miller_accum): the `a`
// operands are the caller's registers (Fp12 coefficients gathered by warp shuffles), the `b` operands are read from shared
// memory four limbs at a time (LDS.128).  Same accumulator shapes as fp_dot6.
__device__ __forceinline__ uint32_t b3_u4_get(const uint4& v, int i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }
// Three terms, for the Karatsuba form of the sparse line product: 3 x 144 + 156 multiply-accumulates.  All operands < 2p:
// the running value stays below (a0 + a1 + a2 + p)(1 + 2^-32) < 7.01p < 2^384, the result below 12p^2/2^384 + p < 2.22p,
// so it ends with one conditional subtraction of 2p.
__device__ __forceinline__ void fp_dot3_rs(fp& r, const fp& a0, const fp& a1, const fp& a2, const fp* b0, const fp* b1, const fp* b2) {
    uint32_t even[12], odd[12];
    const fp* bp[3] = {b0, b1, b2};
#pragma unroll
    for (int q4 = 0; q4 < 3; q4++) {
        uint4 bw[3];
#pragma unroll
        for (int t = 0; t < 3; t++) bw[t] = reinterpret_cast<const uint4*>(bp[t]->l)[q4];
#pragma unroll
        for (int ii = 0; ii < 4; ii++) {
            const int i = 4 * q4 + ii;
            uint32_t* E = (i & 1) ? odd : even;
            uint32_t* O = (i & 1) ? even : odd;
            uint32_t bi = b3_u4_get(bw[0], ii);
            if (i == 0) {
                b3_mul_row(O, a0.l + 1, bi);
                b3_mul_row(E, a0.l, bi);
            } else {
                E[0] = add_cc(E[0], O[1]);
                b3_mad_row_shift(O, a0.l + 1, bi);
                b3_mad_row(E, a0.l, bi);
                O[11] = addc(O[11], 0);
            }
            bi = b3_u4_get(bw[1], ii);
            b3_mad_row(O, a1.l + 1, bi);
            b3_mad_row(E, a1.l, bi);
            O[11] = addc(O[11], 0);
            bi = b3_u4_get(bw[2], ii);
            b3_mad_row(O, a2.l + 1, bi);
            b3_mad_row(E, a2.l, bi);
            O[11] = addc(O[11], 0);
            uint32_t m = E[0] * FP_PINV32;
            b3_mad_row(O, FP_P.l + 1, m);
            b3_mad_row(E, FP_P.l, m);
            O[11] = addc(O[11], 0);
        }
    }
    even[0] = add_cc(even[0], odd[1]);
#pragma unroll
    for (int i = 1; i < 11; i++) even[i] = addc_cc(even[i], odd[i + 1]);
    even[11] = addc(even[11], 0);
    fp_cond_sub(r, even, FP_2P);
}
#endif

#if !defined(B3_HOSTSIM)
// out-of-line form (operands and result in registers): ONE copy of the 588-product body instead of one per call site -- the
// accumulation kernel calls it three times per line and its fully unrolled loop body no longer fit the instruction cache
__device__ __noinline__ fp fp_dot3_rs_v(fp a0, fp a1, fp a2, const fp* b0, const fp* b1, const fp* b2) {
    fp r;
    fp_dot3_rs(r, a0, a1, a2, b0, b1, b2);
    return r;
}
#endif

// Montgomery SQUARING  r = a^2 / 2^384 mod p, r < 2p  (a < 2p), row-wise with the same interleaved reduction as fp_mul_inl, but using
//   a^2 = sum_i a_i 2^(32 i) * ( a_i 2^(32 i) + 2 sum_{j>i} a_j 2^(32 j) ):
// row i adds a_i times the limbs j >= i of that bracket only -- a_i itself at j = i, a_(i+1) << 1 at j = i + 1 and the limbs
// d_j = (a_j << 1) | (a_(j-1) >> 31) of 2a above (2a < 4p < 2^383 has no 13th limb) -- i.e. 12 - i products instead of 12:
// 78 + 144 + 12 = 234 multiply-accumulates instead of 300.  Every contribution to limb k (pairs i + j = k) is added in a
// row min(i, j) <= k, before limb k is reduced, so the interleaved reduction stays valid.  Bounds: the running value
// obeys W' < W / 2^32 + 2a + p, hence W < 5p (1 + 2^-32) < 2^384 as in fp_mul2_inl (same accumulator shapes, same dropped
// carries), and the result (a^2 + m p) / 2^384 < 4p^2/2^384 + p < 1.41p needs no final subtraction.
template <int I>
B3_FN void b3_sqr_row(uint32_t* E, uint32_t* O, const uint32_t* a, const uint32_t* d) {
#define B3_SQW(j) ((j) == I ? a[(j)] : (j) == I + 1 ? (a[(j)] << 1) : d[(j)])
    const uint32_t ai = a[I];
    if (I == 0) {
#pragma unroll
        for (int j = 0; j < 12; j += 2) mul_wide(O[j], O[j + 1], B3_SQW(j + 1), ai);
#pragma unroll
        for (int j = 0; j < 12; j += 2) mul_wide(E[j], E[j + 1], B3_SQW(j), ai);
    } else {
        E[0] = add_cc(E[0], O[1]);
        // O = (O >> 64) + products at the odd window positions >= I, carry in from the addition above
#pragma unroll
        for (int j = 0; j < 10; j += 2) {
            if (j + 1 >= I) madc_wide_cc_in(O[j], O[j + 1], B3_SQW(j + 1), ai, O[j + 2], O[j + 3]);
            else { O[j] = addc_cc(O[j + 2], 0); O[j + 1] = addc_cc(O[j + 3], 0); }
        }
        madc_wide_last(O[10], O[11], B3_SQW(11), ai);                  // position 11 >= I always
        // E += products at the even window positions >= I
        if (I <= 10) {
            const int j0 = (I + 1) & ~1;
            mad_wide_cc(E[j0], E[j0 + 1], B3_SQW(j0), ai);
#pragma unroll
            for (int j = j0 + 2; j < 12; j += 2) madc_wide_cc(E[j], E[j + 1], B3_SQW(j), ai);
            O[11] = addc(O[11], 0);
        }
    }
    uint32_t m = E[0] * FP_PINV32;
    b3_mad_row(O, FP_P.l + 1, m);
    b3_mad_row(E, FP_P.l, m);
    O[11] = addc(O[11], 0);
#undef B3_SQW
}
B3_FN void fp_sqr_inl(fp& r, const fp& a) {
    uint32_t even[12], odd[12], av[12], d[12];
#pragma unroll
    for (int i = 0; i < 12; i++) av[i] = a.l[i];
    d[0] = av[0] << 1;
#pragma unroll
    for (int i = 1; i < 12; i++) d[i] = (av[i] << 1) | (av[i - 1] >> 31);
    b3_sqr_row<0>(even, odd, av, d);  b3_sqr_row<1>(odd, even, av, d);
    b3_sqr_row<2>(even, odd, av, d);  b3_sqr_row<3>(odd, even, av, d);
    b3_sqr_row<4>(even, odd, av, d);  b3_sqr_row<5>(odd, even, av, d);
    b3_sqr_row<6>(even, odd, av, d);  b3_sqr_row<7>(odd, even, av, d);
    b3_sqr_row<8>(even, odd, av, d);  b3_sqr_row<9>(odd, even, av, d);
    b3_sqr_row<10>(even, odd, av, d); b3_sqr_row<11>(odd, even, av, d);
    r.l[0] = add_cc(even[0], odd[1]);
#pragma unroll
    for (int i = 1; i < 11; i++) r.l[i] = addc_cc(even[i], odd[i + 1]);
    r.l[11] = addc(even[11], 0);
}

// Out-of-line multipliers take and return their operands BY VALUE: ptxas then passes them in registers, and the
// callers' field elements never have their address taken, so they stay in registers instead of the local-memory
// stack (by-reference noinline calls put every operand through LDL/STL: 113 M local loads in the first Miller
// kernel, profiles/r1a_miller_full.txt).  The by-reference spellings below are force-inlined shims.
B3_FN_NOINLINE fp fp_mul_v(fp a, fp b) { fp r; fp_mul_inl(r, a, b); return r; }
B3_FN_NOINLINE fp fp_mul2_v(fp a1, fp b1, fp a2, fp b2) { fp r; fp_mul2_inl(r, a1, b1, a2, b2); return r; }
B3_FN void fp_mul2(fp& r, const fp& a1, const fp& b1, const fp& a2, const fp& b2) { r = fp_mul2_v(a1, b1, a2, b2); }
B3_FN void fp_mul(fp& r, const fp& a, const fp& b) { r = fp_mul_v(a, b); }
B3_FN_NOINLINE fp fp_sqr_v(fp a) { fp r; fp_sqr_inl(r, a); return r; }
B3_FN void fp_sqr(fp& r, const fp& a) { r = fp_sqr_v(a); }

// Montgomery form <-> canonical
B3_FN void fp_to_mont(fp& r, const fp& a) { fp_mul(r, FP_R2, a); }       // a any 384-bit value
// (a + mp)/2^384 <= p: only a residue of 0 (a = p) comes out non-canonical, as p
B3_FN void fp_from_mont(fp& r, const fp& a) { fp t; fp_mul(t, a, FP_RAW_ONE); fp_canon(r, t); }

// r = a^e for a fixed public exponent e (plain 384-bit integer): 5-bit SLIDING windows over a table of the odd powers
// a, a^3, .., a^31 (one squaring + 15 multiplications), so a window is spent only on a bit string that starts and ends with
// a one: for e = (p - 3)/4 that is 376 squarings + 66 + 15 multiplications instead of 380 + 90 + 14 with fixed 4-bit windows.
// The exponent is the same in every thread: the control flow is uniform.
B3_FN uint32_t fp_exp_bit(const fp& e, int i) { return (e.l[i >> 5] >> (i & 31)) & 1u; }
B3_FN_NOINLINE void fp_pow_const(fp& r, const fp& a, const fp& e) {
    fp tbl[16];
    fp a2;
    fp_sqr(a2, a);
    tbl[0] = a;
    for (int k = 1; k < 16; k++) fp_mul(tbl[k], tbl[k - 1], a2);
    fp acc = FP_ONE;
    bool started = false;
    int i = 383;
    while (i >= 0 && !fp_exp_bit(e, i)) i--;
    while (i >= 0) {
        if (!fp_exp_bit(e, i)) {
            fp_sqr(acc, acc);
            i--;
            continue;
        }
        int l = i + 1 < 5 ? i + 1 : 5;
        uint32_t w = 0;
        for (int t = 0; t < l; t++) w = (w << 1) | fp_exp_bit(e, i - t);
        while (!(w & 1u)) { w >>= 1; l--; }
        if (started) {
            for (int t = 0; t < l; t++) fp_sqr(acc, acc);
            fp_mul(acc, acc, tbl[w >> 1]);
        } else {
            acc = tbl[w >> 1];
            started = true;
        }
        i -= l;
    }
    r = acc;
}

// canonical integer comparison (inputs are plain 384-bit integers)
B3_FN bool fp_raw_gt(const fp& a, const fp& b) {      // a > b
    uint32_t t = sub_cc(b.l[0], a.l[0]);
#pragma unroll
    for (int i = 1; i < 12; i++) t = subc_cc(b.l[i], a.l[i]);
    (void)t;
    return subc(0, 0) != 0;
}
B3_FN bool fp_raw_is_one(const fp& a) {
    uint32_t t = a.l[0] ^ 1u;
#pragma unroll
    for (int i = 1; i < 12; i++) t |= a.l[i];
    return t == 0;
}
// 1/a mod p (0 -> 0) by the binary extended Euclidean algorithm on the Montgomery representative, about 5x fewer
// instructions than the Fermat exponentiation a^(p-2) the reference uses (A/fp.rs:608-616); the value is the same.
// With abar = a R: the loop yields abar^-1 = a^-1 R^-1 as a plain integer; one multiplication by R^3 gives a^-1 R.
// Data-dependent control flow (the operand is public on this path).  The loop runs on the canonical representative.
B3_FN_NOINLINE void fp_inv(fp& r, const fp& a) {
    fp u, v = FP_P, x1 = FP_RAW_ONE, x2 = FP_NIL;
    fp_canon(u, a);
    if (fp_is_zero(u)) { r = FP_NIL; return; }
    while (!fp_raw_is_one(u) && !fp_raw_is_one(v)) {
        if (!(u.l[0] & 1u)) {
#pragma unroll
            for (int i = 0; i < 11; i++) u.l[i] = (u.l[i] >> 1) | (u.l[i + 1] << 31);
            u.l[11] >>= 1;
            fp_half(x1, x1);
        } else if (!(v.l[0] & 1u)) {
#pragma unroll
            for (int i = 0; i < 11; i++) v.l[i] = (v.l[i] >> 1) | (v.l[i + 1] << 31);
            v.l[11] >>= 1;
            fp_half(x2, x2);
        } else if (fp_raw_gt(u, v)) {
            u.l[0] = sub_cc(u.l[0], v.l[0]);
#pragma unroll
            for (int i = 1; i < 11; i++) u.l[i] = subc_cc(u.l[i], v.l[i]);
            u.l[11] = subc(u.l[11], v.l[11]);
            fp_sub(x1, x1, x2);
        } else {
            v.l[0] = sub_cc(v.l[0], u.l[0]);
#pragma unroll
            for (int i = 1; i < 11; i++) v.l[i] = subc_cc(v.l[i], u.l[i]);
            v.l[11] = subc(v.l[11], u.l[11]);
            fp_sub(x2, x2, x1);
        }
    }
    fp t;
    fp_select(t, fp_raw_is_one(u), x1, x2);
    fp_mul(r, t, FP_R3);
}

// Square root helper for p = 3 mod 4.  Given d, g = d^((p-3)/4):
//   t = g*d, chi = t*g = d^((p-1)/2) in {0, 1, -1}.  If chi == 1: t^2 = d and 1/t = g.
//   If chi == -1: t^2 = -d and 1/t = -g.
// Returns is_qr (chi != -1), t and tinv = g*chi.
B3_FN_NOINLINE bool fp_sqrt_ratio_parts(fp& t, fp& tinv, const fp& d) {
    fp g, chi;
    fp_pow_const(g, d, FP_EXP_SQRT_G);
    fp_mul(t, g, d);
    fp_mul(chi, t, g);
    bool is_one = fp_eq(chi, FP_ONE);
    bool is_zero = fp_is_zero(chi);
    fp ng;
    fp_neg(ng, g);
    fp_select(tinv, is_one, g, ng);
    return is_one || is_zero;
}

// canonical integer comparison helpers (inputs canonical, NOT Montgomery)
B3_FN bool fp_raw_lt_p(const fp& a) { return fp_raw_gt(FP_P, a); }

// ------------------------------------------------------------------------------------------------
// Wire loads / stores, 16 bytes at a time.  Every record of the wire formats is a multiple of 16 bytes (48 / 96 / 192),
// so a 16-byte-aligned array is read with LDG.128 and byte-swapped in registers (PRMT).
// ------------------------------------------------------------------------------------------------
#if defined(B3_HOSTSIM)
struct b3_q16 { uint32_t x, y, z, w; };
static inline uint32_t b3_bswap(uint32_t v) { return __builtin_bswap32(v); }
#else
typedef uint4 b3_q16;
__device__ __forceinline__ uint32_t b3_bswap(uint32_t v) { return __byte_perm(v, 0, 0x0123); }
#endif
B3_FN bool b3_aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
B3_FN void b3_q16_from_bytes(b3_q16& q, const uint8_t* b) {
    q.x = (uint32_t)b[0] | ((uint32_t)b[1] << 8) | ((uint32_t)b[2] << 16) | ((uint32_t)b[3] << 24);
    q.y = (uint32_t)b[4] | ((uint32_t)b[5] << 8) | ((uint32_t)b[6] << 16) | ((uint32_t)b[7] << 24);
    q.z = (uint32_t)b[8] | ((uint32_t)b[9] << 8) | ((uint32_t)b[10] << 16) | ((uint32_t)b[11] << 24);
    q.w = (uint32_t)b[12] | ((uint32_t)b[13] << 8) | ((uint32_t)b[14] << 16) | ((uint32_t)b[15] << 24);
}
B3_FN void b3_q16_to_bytes(uint8_t* b, const b3_q16& q) {
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; i++) { b[4 * i] = (uint8_t)w[i]; b[4 * i + 1] = (uint8_t)(w[i] >> 8); b[4 * i + 2] = (uint8_t)(w[i] >> 16); b[4 * i + 3] = (uint8_t)(w[i] >> 24); }
}
// N16 16-byte words of a wire record.  Device arrays are 16-byte aligned by contract: the host-pointer entries stage into the
// context's own buffers, the *_dev entries reject unaligned pointers (capi.cu: dev_aligned), so the device path is LDG.128 /
// STG.128 only.  The host build (tests/hostsim) takes any pointer.
template <int N16>
B3_FN void wire_load(b3_q16* q, const uint8_t* in) {
#if defined(B3_HOSTSIM)
    for (int i = 0; i < N16; i++) b3_q16_from_bytes(q[i], in + 16 * i);
#else
#pragma unroll
    for (int i = 0; i < N16; i++) q[i] = __ldg(reinterpret_cast<const uint4*>(in) + i);
#endif
}
template <int N16>
B3_FN void wire_store(uint8_t* out, const b3_q16* q) {
#if defined(B3_HOSTSIM)
    for (int i = 0; i < N16; i++) b3_q16_to_bytes(out + 16 * i, q[i]);
#else
#pragma unroll
    for (int i = 0; i < N16; i++) reinterpret_cast<uint4*>(out)[i] = q[i];
#endif
}
// 48 big-endian bytes held as three 16-byte words <-> raw limbs (limb i = byte-swapped word 11 - i); the writer takes a value
// below 2p and emits its canonical representative
B3_FN void fp_raw_from_q(fp& r, const b3_q16* q) {
    r.l[0] = b3_bswap(q[2].w); r.l[1] = b3_bswap(q[2].z); r.l[2] = b3_bswap(q[2].y); r.l[3] = b3_bswap(q[2].x);
    r.l[4] = b3_bswap(q[1].w); r.l[5] = b3_bswap(q[1].z); r.l[6] = b3_bswap(q[1].y); r.l[7] = b3_bswap(q[1].x);
    r.l[8] = b3_bswap(q[0].w); r.l[9] = b3_bswap(q[0].z); r.l[10] = b3_bswap(q[0].y); r.l[11] = b3_bswap(q[0].x);
}
B3_FN void fp_raw_to_q(b3_q16* q, const fp& v) {
    fp a;
    fp_canon(a, v);
    q[2].w = b3_bswap(a.l[0]); q[2].z = b3_bswap(a.l[1]); q[2].y = b3_bswap(a.l[2]); q[2].x = b3_bswap(a.l[3]);
    q[1].w = b3_bswap(a.l[4]); q[1].z = b3_bswap(a.l[5]); q[1].y = b3_bswap(a.l[6]); q[1].x = b3_bswap(a.l[7]);
    q[0].w = b3_bswap(a.l[8]); q[0].z = b3_bswap(a.l[9]); q[0].y = b3_bswap(a.l[10]); q[0].x = b3_bswap(a.l[11]);
}
// OR of the words of n 16-byte words (all-zero test of a record)
B3_FN uint32_t b3_q16_or(const b3_q16* q, int n) {
    uint32_t acc = 0;
#pragma unroll
    for (int i = 0; i < n; i++) acc |= q[i].x | q[i].y | q[i].z | q[i].w;
    return acc;
}
// 48 big-endian bytes <-> raw limbs through a byte pointer (any alignment)
B3_FN void fp_raw_from_be(fp& r, const uint8_t* b) {
    b3_q16 q[3];
    wire_load<3>(q, b);
    fp_raw_from_q(r, q);
}
B3_FN void fp_raw_to_be(uint8_t* b, const fp& a) {
    b3_q16 q[3];
    fp_raw_to_q(q, a);
    wire_store<3>(b, q);
}
