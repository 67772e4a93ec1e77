// TEST INFRASTRUCTURE ONLY.  The field primitives of milagro_bls_b200/csrc/fp.cuh on raw Montgomery residues, compiled for
// the host (B3_HOSTSIM), so that tests/test_hostsim_relaxed.py can feed them non-canonical operands in [p, 2p) and read
// the representative they return without any conversion.  Values cross the interface as 12 little-endian u32 limbs.
#define B3_HOSTSIM 1
#include <string.h>
#include "../../milagro_bls_b200/csrc/fp.cuh"

static fp ld(const uint8_t* b) { fp r; memcpy(r.l, b, 48); return r; }
static void st(uint8_t* b, const fp& a) { memcpy(b, a.l, 48); }

extern "C" {
// op: 0 mul(a, b), 1 sqr(a), 2 mul2(a, b, c, d), 3 add, 4 sub, 5 neg(a), 6 dbl(a), 7 half(a), 8 canon(a), 9 from_mont(a),
//     10 inv(a), 11 wire writer (big-endian bytes), 12 is_zero(a) -> out[0], 13 eq(a, b) -> out[0],
//     14 mul(add_nr(a, b), c), 15 mul2(c, d, neg_nr(a), b), 16 neg_nr(a)
void hs_fp_raw(int op, const uint8_t* a, const uint8_t* b, const uint8_t* c, const uint8_t* d, uint8_t* out) {
    fp x = ld(a), y = ld(b), z = ld(c), w = ld(d), r = FP_NIL;
    switch (op) {
        case 0: fp_mul(r, x, y); break;
        case 1: fp_sqr(r, x); break;
        case 2: fp_mul2(r, x, y, z, w); break;
        case 3: fp_add(r, x, y); break;
        case 4: fp_sub(r, x, y); break;
        case 5: fp_neg(r, x); break;
        case 6: fp_dbl(r, x); break;
        case 7: fp_half(r, x); break;
        case 8: fp_canon(r, x); break;
        case 9: fp_from_mont(r, x); break;
        case 10: fp_inv(r, x); break;
        case 11: fp_raw_to_be(out, x); return;
        case 14: { fp s; fp_add_nr(s, x, y); fp_mul_inl(r, s, z); break; }
        case 15: { fp n; fp_neg_nr(n, x); fp_mul2_inl(r, z, w, n, y); break; }
        case 16: fp_neg_nr(r, x); break;
        case 12: memset(out, 0, 48); out[0] = fp_is_zero(x); return;
        default: memset(out, 0, 48); out[0] = fp_eq(x, y); return;
    }
    st(out, r);
}
// six-term dot product: a = 6 operands, b = 6 operands, each 48 bytes
void hs_fp_dot6_raw(const uint8_t* a, const uint8_t* b, uint8_t* out) {
    fp av[6], bv[6], r;
    fp_dot6_args q;
    for (int t = 0; t < 6; t++) { av[t] = ld(a + 48 * t); bv[t] = ld(b + 48 * t); q.a[t] = &av[t]; q.b[t] = &bv[t]; }
    fp_dot6(r, q);
    st(out, r);
}
}
