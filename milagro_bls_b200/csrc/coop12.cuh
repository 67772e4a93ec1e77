// Cooperative Fp12 arithmetic: ONE CTA (B3_COOP_THREADS threads) works on Fp12 values held in shared memory.
//
// Used where the path is a single long dependent chain of Fp12 operations with nothing else to run beside it:
// the final exponentiation (A/pair.rs:409-541) and the closing sqr/mul chain of the multi-Miller loop
// (A/pair.rs:166-178).  An Fp12 product is done schoolbook over the six Fp2 coefficients of the w-power basis
// (w^6 = xi): 36 Fp2 products, each coordinate of each product ONE dual Montgomery product (fp_mul2) on its own
// thread (72 threads), then 12 threads add up the six terms of the 12 output coordinates.  Latency of an Fp12
// multiplication or squaring is therefore about 1.5 Fp-multiplication latencies plus five additions, instead of 54
// multiplications (18 for a cyclotomic squaring) on one thread.
//
// Every routine is written as per-thread "phase" functions taking an explicit thread index, with a CTA barrier
// between phases, so tests/hostsim can replay the phases sequentially on the CPU.
#pragma once
#include "pairing.cuh"

#define B3_COOP_THREADS 128

struct coop_ws {
    fp val[72];
};

// w-power k (0..5) -> index of that Fp2 coefficient in the memory order of fp12 (c0.c0,c0.c1,c0.c2,c1.c0,c1.c1,c1.c2)
B3_FN int coop_slot(int k) { return (k & 1) ? 3 + (k >> 1) : (k >> 1); }
B3_FN const fp2& coop_coef(const fp12& a, int k) { return reinterpret_cast<const fp2*>(&a)[coop_slot(k)]; }
B3_FN fp2& coop_coef(fp12& a, int k) { return reinterpret_cast<fp2*>(&a)[coop_slot(k)]; }

// ---- r = a * b --------------------------------------------------------------------------------
// r_k = sum_{i+j=k} a_i b_j + xi sum_{i+j=k+6} a_i b_j   (k = 0..5, Fp2 coefficients of w^k).
// phase 1: thread tid < 72 = (output coordinate c = 2k + comp, term i) computes ONE coordinate of ONE term
//   a_i * B,  B = b_j (i + j = k)  or  xi b_j (i + j = k + 6),  as a dual product with a single reduction:
//   comp 0:  a_i0 B0 + (-a_i1) B1        comp 1:  a_i0 B1 + a_i1 B0
B3_FN void coop_mul_p1(coop_ws& ws, const fp12& a, const fp12& b, int tid) {
    if (tid >= 72) return;
    const int c = tid / 6, i = tid - 6 * c, k = c >> 1, comp = c & 1;
    int j = k - i;
    const bool wrap = j < 0;
    if (wrap) j += 6;
    const fp2& x = coop_coef(a, i);
    const fp2& y = coop_coef(b, j);
    fp B0 = y.c0, B1 = y.c1;
    if (wrap) {                                    // xi (y0 + y1 i) = (y0 - y1) + (y0 + y1) i
        fp_sub(B0, y.c0, y.c1);
        fp_add(B1, y.c0, y.c1);
    }
    fp u2, v1, v2;
    fp_neg_nr(u2, x.c1);                           // <= 2p: an operand of the dual product only
    fp_select(u2, comp != 0, x.c1, u2);
    fp_select(v1, comp != 0, B1, B0);
    fp_select(v2, comp != 0, B0, B1);
    fp_mul2(ws.val[tid], x.c0, v1, u2, v2);
}
// phase 2: thread tid < 12 sums the six terms of one output coordinate
B3_FN void coop_mul_p2(fp12& r, const coop_ws& ws, int tid) {
    if (tid >= 12) return;
    fp acc = ws.val[6 * tid];
    for (int i = 1; i < 6; i++) fp_add(acc, acc, ws.val[6 * tid + i]);
    fp2& o = coop_coef(r, tid >> 1);
    if (tid & 1) o.c1 = acc; else o.c0 = acc;
}
// ---- r = conj(a) (w -> -w): odd w-powers negated -----------------------------------------------------------
B3_FN void coop_conj_p(fp12& r, const fp12& a, int tid) {
    if (tid >= 6) return;
    const fp2& x = coop_coef(a, tid);
    fp2 t;
    if (tid & 1) fp2_neg(t, x); else t = x;
    coop_coef(r, tid) = t;
}
// ---- Frobenius maps, one coefficient per thread (n = 1, 2, 3) ------------------------------------------------
B3_FN void coop_frob_p(fp12& r, const fp12& a, int n, int tid) {
    if (tid >= 6) return;
    fp2 t = coop_coef(a, tid), o;
    if (n == 2) {
        if (tid == 0) o = t; else fp2_mul_fp(o, t, FROB_GAMMA2[tid]);
    } else {
        fp2_conj(t, t);
        if (tid == 0) o = t; else fp2_mul(o, t, n == 1 ? FROB_GAMMA1[tid] : FROB_GAMMA3[tid]);
    }
    coop_coef(r, tid) = o;
}
B3_FN void coop_copy_p(fp12& r, const fp12& a, int tid) {
    if (tid >= 12) return;
    reinterpret_cast<fp*>(&r)[tid] = reinterpret_cast<const fp*>(&a)[tid];
}

// A phase: every thread of the CTA runs `stmt` with its index `tid`, then the CTA synchronises.  The host build
// (tests/hostsim) replays the threads of a phase one after another.
#if defined(B3_HOSTSIM)
#define COOP_PHASE(stmt) do { for (int tid = 0; tid < B3_COOP_THREADS; tid++) { stmt; } } while (0)
#define COOP_FN static
#else
#define COOP_PHASE(stmt) do { { const int tid = (int)threadIdx.x; stmt; } __syncthreads(); } while (0)
#define COOP_FN __device__ __noinline__
#endif
// r may alias a and/or b: phase 1 reads a, b; phase 2 reads only ws
COOP_FN void coop_fp12_mul(fp12& r, const fp12& a, const fp12& b, coop_ws& ws) {
    COOP_PHASE(coop_mul_p1(ws, a, b, tid));
    COOP_PHASE(coop_mul_p2(r, ws, tid));
}
COOP_FN void coop_fp12_conj(fp12& r, const fp12& a) { COOP_PHASE(coop_conj_p(r, a, tid)); }
COOP_FN void coop_fp12_frob(fp12& r, const fp12& a, int n) { COOP_PHASE(coop_frob_p(r, a, n, tid)); }   // r must not alias a
COOP_FN void coop_fp12_copy(fp12& r, const fp12& a) { COOP_PHASE(coop_copy_p(r, a, tid)); }
// r = a^(|x| >> shift) by plain square-and-multiply; r must not alias a
COOP_FN void coop_fp12_pow_x_abs(fp12& r, const fp12& a, int shift, coop_ws& ws) {
    const uint64_t x = B3_X_ABS >> shift;
    coop_fp12_copy(r, a);
    for (int i = 62 - shift; i >= 0; i--) {
        coop_fp12_mul(r, r, r, ws);
        if ((x >> i) & 1) coop_fp12_mul(r, r, a, ws);
    }
}
// r = a^x (x negative): pow(|x|) then conjugate
COOP_FN void coop_fp12_pow_x(fp12& r, const fp12& a, int shift, coop_ws& ws) {
    coop_fp12_pow_x_abs(r, a, shift, ws);
    coop_fp12_conj(r, r);
}

// Closing chain of the split Miller loop (pairing.cuh): slots[s] = product over all pairs of the lines of slot s.
//   f = 1; for it = 0..62: f = f^2 * slots[it] [* slots[63 + k] on the addition steps]; f = conj(f)
COOP_FN void coop_miller_chain(fp12& f, const fp12* slots, coop_ws& ws) {
    const uint64_t x = B3_X_ABS;
    int a = B3_MILLER_DBL_SLOTS;
    coop_fp12_copy(f, slots[0]);
    for (int it = 0; it < B3_MILLER_DBL_SLOTS; it++) {
        if (it) {
            coop_fp12_mul(f, f, f, ws);
            coop_fp12_mul(f, f, slots[it], ws);
        }
        if ((x >> (62 - it)) & 1) coop_fp12_mul(f, f, slots[a++], ws);
    }
    coop_fp12_conj(f, f);
}

// ---- r = a * L for a line L = l0 + l3 w^3 + l5 w^5 (dense fp12 whose other coefficients are NOT read) ------------
// r_k = a_k l0 + a_(k-3) l3 + a_(k-5) l5 with xi on the wrapped terms: 18 Fp2 products instead of 36.
// phase 1: thread tid < 36 = (output coordinate c = 2k + comp, term t of {l0, l3, l5})
B3_FN void coop_mul_line_p1(coop_ws& ws, const fp12& a, const fp12& l, int tid) {
    if (tid >= 36) return;
    const int c = tid / 3, t = tid - 3 * c, k = c >> 1, comp = c & 1;
    const int j = t == 0 ? 0 : t == 1 ? 3 : 5;
    int i = k - j;
    const bool wrap = i < 0;
    if (wrap) i += 6;
    const fp2& x = coop_coef(a, i);
    const fp2& y = coop_coef(l, j);
    fp B0 = y.c0, B1 = y.c1;
    if (wrap) {
        fp_sub(B0, y.c0, y.c1);
        fp_add(B1, y.c0, y.c1);
    }
    fp u2, v1, v2;
    fp_neg_nr(u2, x.c1);                           // <= 2p: an operand of the dual product only
    fp_select(u2, comp != 0, x.c1, u2);
    fp_select(v1, comp != 0, B1, B0);
    fp_select(v2, comp != 0, B0, B1);
    fp_mul2(ws.val[tid], x.c0, v1, u2, v2);
}
B3_FN void coop_mul_line_p2(fp12& r, const coop_ws& ws, int tid) {
    if (tid >= 12) return;
    fp acc = ws.val[3 * tid];
    fp_add(acc, acc, ws.val[3 * tid + 1]);
    fp_add(acc, acc, ws.val[3 * tid + 2]);
    fp2& o = coop_coef(r, tid >> 1);
    if (tid & 1) o.c1 = acc; else o.c0 = acc;
}
COOP_FN void coop_fp12_mul_line(fp12& r, const fp12& a, const fp12& l, coop_ws& ws) {
    COOP_PHASE(coop_mul_line_p1(ws, a, l, tid));
    COOP_PHASE(coop_mul_line_p2(r, ws, tid));
}

// ---- Miller product of the few pairs of ONE item, read straight from the line table of the split Miller loop --------
// (batched per-item verification: Signature::verify / fast_aggregate_verify of many independent items, each with its own
// final exponentiation -- the shape of A/pair.rs:313-405 `ate2`, one CTA per item).
struct coop_item_pair {
    size_t idx;            // pair index in the line table
    fp ny, z3, xz;         // factors of the G1 member (g1_pp)
    int valid;             // 0: a member is infinity, the pair contributes 1
    const fp2* lines;      // the pair's own line table of np pairs; null: the table passed to coop_item_miller
    size_t np;
};
// thread tid < 6 scales Fp coordinate tid of the unscaled line (u0, l3, u5) by its factor of P -> coefficient w^0 / w^3 / w^5
B3_FN void coop_line_load_p(fp12& line, const fp2* src, const coop_item_pair& pr, int tid) {
    if (tid >= 6) return;
    const int h = tid >> 1;
    const fp v = reinterpret_cast<const fp*>(src)[tid];
    const fp f = h == 0 ? pr.ny : h == 1 ? pr.z3 : pr.xz;
    fp r;
    fp_mul(r, v, f);
    fp2& o = coop_coef(line, h == 0 ? 0 : h == 1 ? 3 : 5);
    if (tid & 1) o.c1 = r; else o.c0 = r;
}
B3_FN void coop_set_p(fp12& r, bool one, int tid) {      // r = 0 or 1
    if (tid >= 12) return;
    reinterpret_cast<fp*>(&r)[tid] = (one && tid == 0) ? FP_ONE : FP_NIL;
}
// f = conj( prod_pairs f_{|x|,Q}(P) ); `line` is scratch.  lines[(slot * n_pairs + idx) * 3 ..] as written by k_miller_lines
// (or the pair's own table, pr.lines / pr.np).
COOP_FN void coop_item_miller(fp12& f, fp12& line, coop_ws& ws, const fp2* lines, size_t n_pairs, const coop_item_pair* pr, int npr) {
    const uint64_t x = B3_X_ABS;
    bool have = false;                                   // uniform over the CTA
    int a = B3_MILLER_DBL_SLOTS;
    COOP_PHASE(coop_set_p(line, false, tid));
    for (int it = 0; it < B3_MILLER_DBL_SLOTS; it++) {
        if (have) coop_fp12_mul(f, f, f, ws);
        const bool add = (x >> (62 - it)) & 1;
        for (int s = 0; s < (add ? 2 : 1); s++) {
            const size_t slot = s == 0 ? (size_t)it : (size_t)a;
            for (int q = 0; q < npr; q++) {
                if (!pr[q].valid) continue;
                const fp2* tab = pr[q].lines ? pr[q].lines : lines;
                const size_t np = pr[q].lines ? pr[q].np : n_pairs;
                COOP_PHASE(coop_line_load_p(line, tab + (slot * np + pr[q].idx) * 3, pr[q], tid));
                if (have) coop_fp12_mul_line(f, f, line, ws);
                else { coop_fp12_copy(f, line); have = true; }
            }
        }
        if (add) a++;
    }
    if (!have) COOP_PHASE(coop_set_p(f, true, tid));
    coop_fp12_conj(f, f);
}

struct coop_fexp_ws {
    coop_ws ws;
    fp12 m, t, y0, y1, y2, y3, rr;
};
// Final exponentiation, same chain as final_exp() in pairing.cuh (exponent 3 (p^12 - 1) / r), CTA-cooperative.
// in: s.m; out: s.rr
COOP_FN void coop_final_exp(coop_fexp_ws& s) {
    coop_ws& ws = s.ws;
    COOP_PHASE(if (tid == 0) fp12_inv(s.t, s.m));
    coop_fp12_conj(s.rr, s.m);
    coop_fp12_mul(s.rr, s.rr, s.t, ws);              // m^(p^6 - 1)
    coop_fp12_frob(s.t, s.rr, 2);
    coop_fp12_mul(s.rr, s.t, s.rr, ws);              // ^(p^2 + 1)
    coop_fp12_mul(s.y0, s.rr, s.rr, ws);             // y0 = r^2
    coop_fp12_pow_x(s.y1, s.y0, 0, ws);              // y1 = y0^x
    coop_fp12_pow_x(s.y2, s.y1, 1, ws);              // y2 = y1^(x/2)
    coop_fp12_conj(s.y3, s.rr);
    coop_fp12_mul(s.y1, s.y1, s.y3, ws);
    coop_fp12_conj(s.y1, s.y1);
    coop_fp12_mul(s.y1, s.y1, s.y2, ws);
    coop_fp12_pow_x(s.y2, s.y1, 0, ws);
    coop_fp12_pow_x(s.y3, s.y2, 0, ws);
    coop_fp12_conj(s.y1, s.y1);
    coop_fp12_mul(s.y3, s.y3, s.y1, ws);
    coop_fp12_conj(s.y1, s.y1);
    coop_fp12_frob(s.t, s.y1, 3);                    // t  = frob3(y1)
    coop_fp12_frob(s.y1, s.y2, 2);                   // y1 = frob2(y2)
    coop_fp12_mul(s.y1, s.t, s.y1, ws);              // y1 = frob3(y1) * frob2(y2)
    coop_fp12_pow_x(s.y2, s.y3, 0, ws);
    coop_fp12_mul(s.y2, s.y2, s.y0, ws);
    coop_fp12_mul(s.y2, s.y2, s.rr, ws);
    coop_fp12_mul(s.y1, s.y1, s.y2, ws);
    coop_fp12_frob(s.y2, s.y3, 1);
    coop_fp12_mul(s.rr, s.y1, s.y2, ws);
}
