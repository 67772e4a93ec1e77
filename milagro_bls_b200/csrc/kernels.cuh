// __global__ kernels of the verification path (sm_100a).  One thread (or one lane group) per item; all field
// arithmetic comes from fp.cuh / tower.cuh / curve.cuh / pairing.cuh / h2c.cuh.
#pragma once
#include "h2c.cuh"
#include "pairing.cuh"
#include "coop12.cuh"
#include "fp2h.cuh"
#include "quad.cuh"

#define B3_ERR_AGGREGATE_EMPTY_POINTS_D (-1)
#define B3_ERR_INVALID_G1_SIZE_D (-6)
#define B3_ERR_INVALID_G2_SIZE_D (-7)

#define B3_TPB 128
#ifndef B3_MIN_CTAS
#define B3_MIN_CTAS 2
#endif
#define B3_LBH __launch_bounds__(B3_TPB, B3_MIN_CTAS)
#ifndef B3_H2C_CTAS
#define B3_H2C_CTAS 2
#endif

// ------------------------------------------------------------------------------------------------ parsing
// G1 uncompressed wire -> Jacobian (Z = 1, or infinity).  status: per-item AmclError code.
__global__ void __launch_bounds__(B3_TPB) k_g1_parse(const uint8_t* __restrict__ in, size_t n, g1_jac* out, int32_t* status, int check_curve) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_aff a;
    int e = g1_aff_from_wire(a, in + 96 * i);
    if (e == B3_OK && check_curve && !pt_on_curve_aff(a)) e = B3_ERR_INVALID_POINT;
    g1_jac j;
    if (e) pt_set_inf(j); else pt_from_aff(j, a);
    out[i] = j;
    status[i] = e;
}
// G2 uncompressed wire -> affine struct; optional on-curve check
__global__ void __launch_bounds__(B3_TPB) k_g2_parse(const uint8_t* __restrict__ in, size_t n, g2_aff* out, int32_t* status, int check_curve) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g2_aff a;
    int e = g2_aff_from_wire(a, in + 192 * i);
    if (e == B3_OK && check_curve && !pt_on_curve_aff(a)) e = B3_ERR_INVALID_POINT;
    if (e) { fp2_zero(a.x); fp2_zero(a.y); a.inf = 1; }
    out[i] = a;
    status[i] = e;
}
// subgroup_check_g2 on parsed signatures: ok[i] = parsed fine && in G2 (infinity passes, SURVEY.md C.4).
// LANE PAIRS (fp2h.cuh): threads (2i, 2i+1) work on signature i.
__global__ void B3_LBH k_g2_subgroup(const g2_aff* pts, const int32_t* status, size_t n, int32_t* ok) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    int good = 0;
    if (status[i] == B3_OK) {
        g2h_aff a;
        g2h_load(a, pts[i]);
        good = g2_in_subgroup_aff(a) ? 1 : 0;
    }
    if (!pair_odd()) ok[i] = good;
}
// the same on LANE QUADS (quad.cuh): threads 4i .. 4i+3 work on signature i, paired products split over the two lane pairs
__global__ void B3_LBH k_g2_subgroup_q(const g2_aff* pts, const int32_t* status, size_t n, int32_t* ok) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    if (i >= n) return;
    int good = 0;
    if (status[i] == B3_OK) {
        g2q_aff a;
        g2q_load(a, pts[i]);
        good = g2_in_subgroup_aff(a) ? 1 : 0;
    }
    if ((threadIdx.x & 3u) == 0) ok[i] = good;
}
// key_validate on parsed G1 points (not infinity, in G1)
__global__ void __launch_bounds__(B3_TPB) k_g1_key_validate(const g1_jac* pts, const int32_t* status, size_t n, int32_t* valid) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_jac p = pts[i];
    valid[i] = (status[i] == B3_OK && !pt_is_inf(p) && g1_in_subgroup(p)) ? 1 : 0;
}

// ------------------------------------------------------------------------------------------------ (de)compression
// Records are read and written as 16-byte words (wire_load / wire_store: LDG.128 / STG.128 on aligned arrays).
template <int N16>
__device__ __forceinline__ void q16_zero(b3_q16* q) {
#pragma unroll
    for (int i = 0; i < N16; i++) { q[i].x = 0; q[i].y = 0; q[i].z = 0; q[i].w = 0; }
}
// ZCash-compressed G1 record (three 16-byte words) -> affine point, optional key_validate (M/src/keys.rs:140-147,181-186)
__device__ __noinline__ int g1_decompress_q(g1_aff& a, const b3_q16* qin, int validate) {
    int e = B3_OK;
    a.x = FP_NIL; a.y = FP_NIL; a.inf = 1;
    b3_q16 q[3] = {qin[0], qin[1], qin[2]};
    const uint32_t b0 = q[0].x & 0xffu;
    if (!(b0 & 0x80)) e = B3_ERR_INVALID_G1_SIZE_D;          // 48 bytes without the C flag: routed to the 96-byte parser
    else if (b0 & 0x40) {
        if ((q[0].x & 0xffffff3fu) | q[0].y | q[0].z | q[0].w | b3_q16_or(q + 1, 2)) e = B3_ERR_INVALID_POINT;
    } else {
        q[0].x &= 0xffffff1fu;
        fp x;
        fp_raw_from_q(x, q);
        if (!fp_raw_lt_p(x)) e = B3_ERR_INVALID_POINT;
        else {
            fp xm, rhs, t, y, yinv;
            fp_to_mont(xm, x);
            fp_sqr(t, xm);
            fp_mul(rhs, t, xm);
            fp_add(t, FP_ONE, FP_ONE);
            fp_dbl(t, t);
            fp_add(rhs, rhs, t);
            bool qr = fp_sqrt_ratio_parts(y, yinv, rhs);
            if (!qr || fp_is_zero(rhs)) e = B3_ERR_INVALID_POINT;
            else {
                fp yc, ny, nyc;
                fp_neg(ny, y);
                fp_from_mont(yc, y);
                fp_from_mont(nyc, ny);
                bool greater = fp_raw_gt(yc, nyc);
                bool yflag = (b0 & 0x20) != 0;
                a.x = xm;
                fp_select(a.y, greater == yflag, y, ny);
                a.inf = 0;
            }
        }
    }
    if (e == B3_OK && validate) {
        g1_jac j;
        pt_from_aff(j, a);
        if (a.inf || !g1_in_subgroup(j)) e = B3_ERR_INVALID_POINT;
    }
    return e;
}
__global__ void __launch_bounds__(B3_TPB) k_g1_decompress(const uint8_t* __restrict__ in, size_t n, int validate, uint8_t* out, int32_t* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t* o = out + 96 * i;
    g1_aff a;
    b3_q16 q[3];
    wire_load<3>(q, in + 48 * i);
    const int e = g1_decompress_q(a, q, validate);
    if (e) { b3_q16 z[6]; q16_zero<6>(z); wire_store<6>(o, z); }
    else g1_aff_to_wire(o, a);
    status[i] = e;
}

// ---- device-resident public-key table (SURVEY.md 8(f)1; the reference pays PublicKey::from_bytes -- decompression + key_validate,
// M/src/keys.rs:140-147 -- once per validator and then aggregates the decoded points, M/src/aggregates.rs:29-39) ----------------
// Entry = (x, y) in Montgomery form, 96 bytes, read with six LDG.128 and used as is: no byte swap, no conversion, no checks per
// use.  Coordinates are stored canonical.  (0, 0) encodes infinity (it is not on the curve); x.l[11] = 0xffffffff (> 2p) marks
// an entry whose input was rejected.
struct key_entry {
    fp x, y;
};
#define B3_KEY_INVALID 0xffffffffu
__global__ void __launch_bounds__(B3_TPB) k_keytable_build(const uint8_t* __restrict__ in, size_t n, int compressed, int validate, key_entry* out,
                                                           int32_t* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_aff a;
    int e;
    if (compressed) {
        b3_q16 q[3];
        wire_load<3>(q, in + 48 * i);
        e = g1_decompress_q(a, q, validate);
    } else {
        e = g1_aff_from_wire(a, in + 96 * i);
        if (e == B3_OK && !pt_on_curve_aff(a)) e = B3_ERR_INVALID_POINT;
        if (e == B3_OK && validate) {
            g1_jac j;
            pt_from_aff(j, a);
            if (a.inf || !g1_in_subgroup(j)) e = B3_ERR_INVALID_POINT;
        }
    }
    key_entry k;
    if (e) { k.x = FP_NIL; k.y = FP_NIL; k.x.l[11] = B3_KEY_INVALID; }
    else if (a.inf) { k.x = FP_NIL; k.y = FP_NIL; }
    else { fp_canon(k.x, a.x); fp_canon(k.y, a.y); }
    out[i] = k;
    status[i] = e;
}
__device__ __forceinline__ void key_entry_load(key_entry& k, const key_entry* p) {
    const uint4* s = reinterpret_cast<const uint4*>(p);
    uint4* d = reinterpret_cast<uint4*>(&k);
#pragma unroll
    for (int j = 0; j < 6; j++) d[j] = __ldg(s + j);
}
// table entry -> affine point; returns B3_ERR_INVALID_POINT for a rejected entry
__device__ __forceinline__ int key_entry_point(g1_aff& a, const key_entry& k) {
    if (k.x.l[11] == B3_KEY_INVALID) return B3_ERR_INVALID_POINT;
    a.x = k.x; a.y = k.y;
    a.inf = (fp_is_zero(k.x) && fp_is_zero(k.y)) ? 1u : 0u;
    return B3_OK;
}
__global__ void __launch_bounds__(B3_TPB) k_keytable_get(const key_entry* __restrict__ table, size_t n_table, const uint32_t* __restrict__ idx, size_t n,
                                                         uint8_t* out96, int32_t* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint32_t k = idx[i];
    g1_aff a;
    a.x = FP_NIL; a.y = FP_NIL; a.inf = 1;
    int e = B3_ERR_INVALID_POINT;
    if (k < n_table) {
        key_entry ent;
        key_entry_load(ent, table + k);
        e = key_entry_point(a, ent);
    }
    if (e) { b3_q16 z[6]; q16_zero<6>(z); wire_store<6>(out96 + 96 * i, z); }
    else g1_aff_to_wire(out96 + 96 * i, a);
    status[i] = e;
}

__global__ void __launch_bounds__(B3_TPB) k_g2_decompress(const uint8_t* __restrict__ in, size_t n, uint8_t* out, int32_t* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint8_t* o = out + 192 * i;
    int e = B3_OK;
    g2_aff a;
    fp2_zero(a.x); fp2_zero(a.y); a.inf = 1;
    b3_q16 q[6];
    wire_load<6>(q, in + 96 * i);
    const uint32_t b0 = q[0].x & 0xffu;
    if (!(b0 & 0x80)) e = B3_ERR_INVALID_G2_SIZE_D;
    else if (b0 & 0x40) {
        if ((q[0].x & 0xffffff3fu) | q[0].y | q[0].z | q[0].w | b3_q16_or(q + 1, 5)) e = B3_ERR_INVALID_POINT;
    } else {
        q[0].x &= 0xffffff1fu;
        fp xim, xre;
        fp_raw_from_q(xim, q);
        fp_raw_from_q(xre, q + 3);
        if (!fp_raw_lt_p(xim) || !fp_raw_lt_p(xre)) e = B3_ERR_INVALID_POINT;
        else {
            fp2 x, rhs, t, y;
            fp_to_mont(x.c0, xre);
            fp_to_mont(x.c1, xim);
            fp2_sqr(t, x);
            fp2_mul(rhs, t, x);
            fp2_one(t);
            f_mul_b(t, t);
            fp2_add(rhs, rhs, t);
            bool sq = fp2_sqrt_or_z(y, rhs);
            // The reference's FP2::sqrt (A/fp2.rs:304-339) also fails on (a0, 0) with a0 a non-residue of Fp,
            // although such elements are squares in Fp2; replicate so accept/reject is bit-exact.
            if (sq && fp_is_zero(rhs.c1) && !fp_is_zero(rhs.c0)) {
                fp s, sinv;
                if (!fp_sqrt_ratio_parts(s, sinv, rhs.c0)) sq = false;
            }
            if (!sq) e = B3_ERR_INVALID_POINT;
            else {
                fp2 ny;
                fp2_neg(ny, y);
                fp yi, yr, nyi, nyr;
                fp_from_mont(yi, y.c1); fp_from_mont(yr, y.c0);
                fp_from_mont(nyi, ny.c1); fp_from_mont(nyr, ny.c0);
                bool greater = fp_raw_gt(yi, nyi) || (fp_eq(yi, nyi) && fp_raw_gt(yr, nyr));
                bool yflag = (b0 & 0x20) != 0;
                a.x = x;
                fp2_select(a.y, greater == yflag, y, ny);
                a.inf = 0;
            }
        }
    }
    if (e) { b3_q16 z[12]; q16_zero<12>(z); wire_store<12>(o, z); }
    else g2_aff_to_wire(o, a);
    status[i] = e;
}

__global__ void __launch_bounds__(B3_TPB) k_g1_compress(const uint8_t* __restrict__ in, size_t n, uint8_t* out, int32_t* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_aff a;
    int e = g1_aff_from_wire(a, in + 96 * i);
    status[i] = e;
    b3_q16 q[3];
    q16_zero<3>(q);
    if (e == B3_OK) {
        if (a.inf) q[0].x = 0xc0;
        else {
            fp xc, yc, ny, nyc;
            fp_from_mont(xc, a.x);
            fp_from_mont(yc, a.y);
            fp_neg(ny, a.y);
            fp_from_mont(nyc, ny);
            fp_raw_to_q(q, xc);
            q[0].x |= 0x80u | (fp_raw_gt(yc, nyc) ? 0x20u : 0u);
        }
    }
    wire_store<3>(out + 48 * i, q);
}
__global__ void __launch_bounds__(B3_TPB) k_g2_compress(const uint8_t* __restrict__ in, size_t n, uint8_t* out, int32_t* status) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g2_aff a;
    int e = g2_aff_from_wire(a, in + 192 * i);
    status[i] = e;
    b3_q16 q[6];
    q16_zero<6>(q);
    if (e == B3_OK) {
        if (a.inf) q[0].x = 0xc0;
        else {
            fp t, yi, yr, nyi, nyr;
            fp2 ny;
            fp2_neg(ny, a.y);
            fp_from_mont(t, a.x.c1); fp_raw_to_q(q, t);
            fp_from_mont(t, a.x.c0); fp_raw_to_q(q + 3, t);
            fp_from_mont(yi, a.y.c1); fp_from_mont(yr, a.y.c0);
            fp_from_mont(nyi, ny.c1); fp_from_mont(nyr, ny.c0);
            bool greater = fp_raw_gt(yi, nyi) || (fp_eq(yi, nyi) && fp_raw_gt(yr, nyr));
            q[0].x |= 0x80u | (greater ? 0x20u : 0u);
        }
    }
    wire_store<6>(out + 96 * i, q);
}

// ------------------------------------------------------------------------------------------------ aggregation
// G1 public-key aggregation: a group of G lanes (G | 32) per set.  Each lane folds its strided share of the keys
// with mixed additions, then the G partial sums are combined by a shuffle tree of Jacobian additions.
template <class P>
__device__ __forceinline__ void shfl_down_struct(P& dst, const P& src, int delta, int width) {
    const uint32_t* s = reinterpret_cast<const uint32_t*>(&src);
    uint32_t* d = reinterpret_cast<uint32_t*>(&dst);
#pragma unroll 1
    for (int k = 0; k < (int)(sizeof(P) / 4); k++) d[k] = __shfl_down_sync(0xffffffffu, s[k], delta, width);
}

// The keys are the bulk of the input bytes (C4: 100 MB of 103 MB), so they are STAGED: the G lanes of a group fetch the group's
// next run of G consecutive 96-byte records as 16-byte words, lane l taking words l, l + G, ... (LDG.128, each warp request
// covering 8 x G*16 contiguous bytes), one step AHEAD of the additions (the loads of step t + 1 are in flight while the
// mixed additions of step t execute); the words pass through shared memory to reach the lane that owns the record.
// check_curve: reject keys that are not on the curve (the reference's types cannot hold such a point: every constructor
// of PublicKey checks, M/src/keys.rs:140-175; pt_add_aff never uses the curve constant, so an unchecked key would
// silently run the arithmetic on another curve).
template <int G>
__global__ void __launch_bounds__(B3_TPB) k_g1_aggregate(const uint8_t* __restrict__ pks, const uint32_t* __restrict__ off, size_t n_sets,
                                                         g1_jac* out, int32_t* status, int check_curve) {
    __shared__ b3_q16 stage[B3_TPB * 6];                    // one 96-byte record per thread
    size_t gid = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const int lane = threadIdx.x % G;
    bool active = gid < n_sets;
    uint32_t b = 0, e = 0;
    if (active) { b = off[gid]; e = off[gid + 1]; }
    b3_q16* const run = stage + (size_t)(threadIdx.x - lane) * 6;
    const uint4* const base16 = reinterpret_cast<const uint4*>(pks);
    g1_jac acc;
    pt_set_inf(acc);
    int err = 0;
    b3_q16 nxt[6];
    uint32_t i0 = b;
    // fetch the run [i0, i0 + G) of this group (clipped to the set): this lane takes words lane, lane + G, ..
#define B3_AGG_FETCH()                                                                                          \
    do {                                                                                                        \
        const uint32_t recs = i0 < e ? (e - i0 < (uint32_t)G ? e - i0 : (uint32_t)G) : 0u;                      \
        _Pragma("unroll") for (int j = 0; j < 6; j++) {                                                         \
            const uint32_t w = (uint32_t)lane + (uint32_t)G * j;                                                \
            if (w < recs * 6) nxt[j] = __ldg(base16 + (size_t)i0 * 6 + w);                                      \
        }                                                                                                       \
    } while (0)
    B3_AGG_FETCH();
    while (__any_sync(0xffffffffu, i0 < e)) {              // warp-uniform trip count (ragged sets): the staging syncs the warp
        b3_q16 q[6];
#pragma unroll
        for (int j = 0; j < 6; j++) run[lane + G * j] = nxt[j];
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 6; j++) q[j] = run[lane * 6 + j];
        __syncwarp();
        const bool mine = i0 < e && i0 + lane < e;
        if (i0 < e) i0 += G;
        B3_AGG_FETCH();
        if (mine) {
            g1_aff a;
            int s = g1_aff_from_q(a, q);
            if (s == B3_OK && check_curve && !pt_on_curve_aff(a)) s = B3_ERR_INVALID_POINT;
            if (s) err = s;
            else pt_add_aff(acc, acc, a);
        }
    }
#undef B3_AGG_FETCH
#pragma unroll 1
    for (int d = G / 2; d >= 1; d >>= 1) {
        g1_jac o;
        shfl_down_struct(o, acc, d, G);
        int oe = __shfl_down_sync(0xffffffffu, err, d, G);
        if (lane < d) {
            pt_add(acc, acc, o);
            if (oe) err = oe;
        }
    }
    if (active && lane == 0) {
        if (b == e) err = B3_ERR_AGGREGATE_EMPTY_POINTS_D;
        out[gid] = acc;
        status[gid] = err;
    }
}
// The same aggregation over a device-resident key table: set s owns the table entries idx[off[s] .. off[s+1]).  A gather of
// 96-byte entries (three full 32-byte sectors each), the next entry in flight while the current one is added.
template <int G>
__global__ void __launch_bounds__(B3_TPB) k_g1_aggregate_idx(const key_entry* __restrict__ table, size_t n_table, const uint32_t* __restrict__ idx,
                                                             const uint32_t* __restrict__ off, size_t n_sets, g1_jac* out, int32_t* status) {
    size_t gid = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    const int lane = threadIdx.x % G;
    bool active = gid < n_sets;
    uint32_t b = 0, e = 0;
    if (active) { b = off[gid]; e = off[gid + 1]; }
    g1_jac acc;
    pt_set_inf(acc);
    int err = 0;
    uint32_t i = b + lane;
    bool have = i < e, ok = false;
    key_entry cur, nxt;
    if (have) {
        const uint32_t k = idx[i];
        ok = k < n_table;
        if (ok) key_entry_load(cur, table + k);
    }
    while (have) {
        const uint32_t inext = i + G;
        const bool hn = inext < e;
        bool okn = false;
        if (hn) {
            const uint32_t k = idx[inext];
            okn = k < n_table;
            if (okn) key_entry_load(nxt, table + k);
        }
        g1_aff a;
        int s = ok ? key_entry_point(a, cur) : B3_ERR_INVALID_POINT;
        if (s) err = s;
        else pt_add_aff(acc, acc, a);
        cur = nxt; ok = okn; have = hn; i = inext;
    }
#pragma unroll 1
    for (int d = G / 2; d >= 1; d >>= 1) {
        g1_jac o;
        shfl_down_struct(o, acc, d, G);
        int oe = __shfl_down_sync(0xffffffffu, err, d, G);
        if (lane < d) {
            pt_add(acc, acc, o);
            if (oe) err = oe;
        }
    }
    if (active && lane == 0) {
        if (b == e) err = B3_ERR_AGGREGATE_EMPTY_POINTS_D;
        out[gid] = acc;
        status[gid] = err;
    }
}
// G2 aggregation (AggregateSignature::aggregate): same shape over Fp2 (records read as 12 x LDG.128 per lane)
template <int G>
__global__ void __launch_bounds__(B3_TPB) k_g2_aggregate(const uint8_t* __restrict__ sigs, const uint32_t* __restrict__ off, size_t n_sets,
                                                         g2_jac* out, int32_t* status, int check_curve) {
    size_t gid = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) / G;
    int lane = threadIdx.x % G;
    bool active = gid < n_sets;
    uint32_t b = 0, e = 0;
    if (active) { b = off[gid]; e = off[gid + 1]; }
    g2_jac acc;
    pt_set_inf(acc);
    int err = 0;
    for (uint32_t i = b + lane; i < e; i += G) {
        g2_aff a;
        int s = g2_aff_from_wire(a, sigs + 192 * (size_t)i);
        if (s == B3_OK && check_curve && !pt_on_curve_aff(a)) s = B3_ERR_INVALID_POINT;
        if (s) err = s;
        else pt_add_aff(acc, acc, a);
    }
#pragma unroll 1
    for (int d = G / 2; d >= 1; d >>= 1) {
        g2_jac o;
        shfl_down_struct(o, acc, d, G);
        int oe = __shfl_down_sync(0xffffffffu, err, d, G);
        if (lane < d) {
            pt_add(acc, acc, o);
            if (oe) err = oe;
        }
    }
    if (active && lane == 0) {
        out[gid] = acc;
        status[gid] = err;
    }
}

// ------------------------------------------------------------------------------------------------ scalar multiplication
// [c_j] sig_j, LANE PAIRS: threads (2i, 2i+1) work on signature i
__global__ void __launch_bounds__(B3_TPB) k_g2_mul_u64(const g2_aff* in, const uint64_t* __restrict__ k, size_t n, g2_jac* out) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    g2h_aff p;
    g2h_load(p, in[i]);
    g2h_jac r;
    pt_mul_u64_aff(r, p, k[i]);
    g2h_store(out[i], r);
}
// 256-bit scalars (32-byte big-endian) -- input synthesis only
__device__ __forceinline__ void load_scalar256(uint32_t* k, const uint8_t* b) {
    b3_q16 q[2];
    wire_load<2>(q, b);
    k[0] = b3_bswap(q[1].w); k[1] = b3_bswap(q[1].z); k[2] = b3_bswap(q[1].y); k[3] = b3_bswap(q[1].x);
    k[4] = b3_bswap(q[0].w); k[5] = b3_bswap(q[0].z); k[6] = b3_bswap(q[0].y); k[7] = b3_bswap(q[0].x);
}
__global__ void __launch_bounds__(B3_TPB) k_g1_mul_gen_u256(const uint8_t* __restrict__ scalars, size_t n, uint8_t* out96) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t k[8];
    load_scalar256(k, scalars + 32 * i);
    g1_aff g;
    g.x = G1_GEN_X; g.y = G1_GEN_Y; g.inf = 0;
    g1_jac r;
    pt_mul_u256_aff(r, g, k);
    g1_aff a;
    pt_to_aff(a, r);
    g1_aff_to_wire(out96 + 96 * i, a);
}
__global__ void __launch_bounds__(B3_TPB) k_g2_mul_u256(const uint8_t* __restrict__ pts, const uint8_t* __restrict__ scalars, size_t n, uint8_t* out192) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    uint32_t k[8];
    load_scalar256(k, scalars + 32 * i);
    g2_aff p;
    int e = g2_aff_from_wire(p, pts + 192 * i);
    if (e) { fp2_zero(p.x); fp2_zero(p.y); p.inf = 1; }
    g2_jac r;
    pt_mul_u256_aff(r, p, k);
    g2_aff a;
    pt_to_aff(a, r);
    g2_aff_to_wire(out192 + 192 * i, a);
}

// ---- S = sum_j [c_j] sig_j as a multi-scalar multiplication (bucket method) -----------------------------------------
// 64-bit scalars, B3_MSM_WINDOWS windows of 8 bits, buckets 1..255 per window (digit 0 adds nothing).
//   1. k_msm_sort : per window, a stable counting sort of the set indices by digit -> idx[w][pos], bucket starts
//   2. k_msm_walk : W_w = sum_b b B_b = sum_b R_b with R_b = sum_(b' >= b) B_b' (running sums), cut into ranges
//   3. k_g2_add_pairs levels: the ranges of a window summed by a pairwise tree
// and the windows are NOT recombined in G2 (56 dependent doublings): by bilinearity
//   e(S, -G1) = prod_w e(W_w, -[2^(8w)] G1)
// so the eight window sums become eight pairs of the multi-Miller loop against precomputed multiples of the
// generator (G1_POW256_*).  The GT value is identical.
#define B3_MSM_WINDOWS 8
#define B3_MSM_BUCKETS 255
// Target events per range of k_msm_walk (the actual length is 0.5x - 1x of this).  A range costs at most q point additions
// whatever the digits: a signature event is one mixed addition (7M + 4S), and where STEPs follow each other (the empty
// buckets around one full bucket when all scalars are equal) every STEP flushes the previous snapshot, one full addition
// (11M + 5S) -- so a step-heavy range costs at most ~1.4x a signature-heavy one.
#define B3_MSM_STEP 96
// idx[w * n + pos]: the set indices ordered by the w-th digit, ties by index (a stable sort, so the order and with it every
// value downstream is the same from run to run); start[w * 257 + d] = first position of digit d, start[w * 257 + 256] = n.
// One CTA per window: a histogram, its scan, then 1024-set tiles ranked by __match_any_sync inside each warp and by a
// column scan of the per-warp digit counts across the tile.
__global__ void __launch_bounds__(1024) k_msm_sort(const uint64_t* __restrict__ k, size_t n, uint32_t* __restrict__ idx, uint32_t* __restrict__ start) {
    __shared__ uint32_t run[256];
    __shared__ uint32_t cnt[32][256];
    const unsigned w = blockIdx.x, tid = threadIdx.x, lane = tid & 31u, warp = tid >> 5, sh = 8 * w;
    uint32_t* st = start + (size_t)w * 257;
    uint32_t* out = idx + (size_t)w * n;
    if (tid < 256) run[tid] = 0;
    __syncthreads();
    for (size_t j = tid; j < n; j += 1024) atomicAdd(&run[(unsigned)(k[j] >> sh) & 255u], 1u);
    __syncthreads();
    if (warp == 0) {                                 // exclusive scan of the 256 counts, 8 per lane
        uint32_t c[8], s = 0;
        for (int i = 0; i < 8; i++) { c[i] = run[lane * 8 + i]; s += c[i]; }
        uint32_t x = s;
        for (unsigned d = 1; d < 32; d <<= 1) {
            const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
            if (lane >= d) x += y;
        }
        uint32_t base = x - s;
        for (int i = 0; i < 8; i++) { run[lane * 8 + i] = base; st[lane * 8 + i] = base; base += c[i]; }
        if (lane == 31) st[256] = base;
    }
    __syncthreads();
    for (size_t t0 = 0; t0 < n; t0 += 1024) {
        for (unsigned i = tid; i < 32 * 256; i += 1024) (&cnt[0][0])[i] = 0;
        __syncthreads();
        const size_t j = t0 + tid;
        const bool live = j < n;
        const unsigned d = live ? (unsigned)(k[j] >> sh) & 255u : 256u;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const unsigned rank = __popc(peers & ((1u << lane) - 1u));
        if (live && rank == 0) cnt[warp][d] = __popc(peers);
        __syncthreads();
        if (tid < 256) {                             // digit tid: where each warp's sets of this digit go
            uint32_t s = run[tid];
            for (int v = 0; v < 32; v++) { const uint32_t c = cnt[v][tid]; cnt[v][tid] = s; s += c; }
            run[tid] = s;
        }
        __syncthreads();
        if (live) out[cnt[warp][d] + rank] = (uint32_t)j;
        __syncthreads();
    }
}
// Ranges of the running-sum walk.  A window's walk is a list of EVENTS, bucket b = 255 down to 1: the signatures of bucket b
// (R += sig), then one STEP (T += R); at the end T = sum_b R_b = W_w.  The list has n - start[1] + 255 <= n + 255 events;
// it is cut into msm_ranges(n) ranges (a power of two, so that the pairwise tree never pairs two windows) of msm_step(n)
// events, one lane pair each: work per lane pair is bounded whatever the digits are (all sets in one bucket is the same
// number of events as random scalars).
__host__ __device__ __forceinline__ unsigned msm_ranges(size_t n) {
    const size_t want = (n + B3_MSM_BUCKETS + B3_MSM_STEP - 1) / B3_MSM_STEP;
    unsigned r = 1;
    while (r < want) r <<= 1;
    return r;
}
__host__ __device__ __forceinline__ unsigned msm_step(size_t n) { return (unsigned)((n + B3_MSM_BUCKETS + msm_ranges(n) - 1) / msm_ranges(n)); }
// Lane pair (w, r) walks events [r q, r q + q) from zero with its own R and T.  The events before it hold the R_before of the
// signatures already added, and each STEP of this range and after it would have added R_before too: out = T + [m] R + ...
// with m = the number of STEPs from the range's end on (= the bucket the next event belongs to), summed over all ranges:
// out[w * nr + r] = T_r + [m_r] R_r, and W_w = sum_r out[w * nr + r].
// The signature additions run in lock step across the warp; a STEP only snapshots R, and the snapshots are added to T
// warp-wide when some pair would need a second one (a branch taken by one pair costs the whole warp its full time).
__global__ void B3_LBH k_msm_walk(const g2_aff* __restrict__ sigs, const uint32_t* __restrict__ idx, const uint32_t* __restrict__ start,
                                  size_t n, unsigned nr, unsigned q, g2_jac* out) {
    const size_t id = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    const bool live = id < (size_t)B3_MSM_WINDOWS * nr;
    const unsigned w = live ? (unsigned)(id / nr) : 0, r = (unsigned)(id % nr);
    const uint32_t* st = start + (size_t)w * 257;
    const uint32_t* ix = idx + (size_t)w * n;
    const size_t total = n - st[1] + B3_MSM_BUCKETS;
    size_t e = (size_t)r * q;
    const size_t e1 = live && e < total ? (e + q < total ? e + q : total) : e;
    // the event e: bucket b = the smallest b >= 1 whose block starts at or before e; blocks start at n - st[b + 1] + 255 - b
    unsigned b = 0;
    size_t pos = 0, end = 0;
    if (e < e1) {
        unsigned lo = 1, hi = B3_MSM_BUCKETS;
        while (lo < hi) {
            const unsigned mid = (lo + hi) >> 1;
            if (n - st[mid + 1] + B3_MSM_BUCKETS - mid <= e) hi = mid; else lo = mid + 1;
        }
        b = lo;
        end = st[b + 1];
        pos = st[b] + (e - (n - end + B3_MSM_BUCKETS - b));
    }
    g2h_jac R, T, S;
    pt_set_inf(R);
    pt_set_inf(T);
    bool pend = false;
    for (unsigned t = 0; t < q; t++, e++) {
        const bool ev = e < e1;
        const bool step = ev && pos == end;
        if (__any_sync(0xffffffffu, step && pend)) {
            if (pend) pt_add(T, T, S);
            pend = false;
        }
        if (step) {
            S = R;
            pend = true;
            b--;
            pos = st[b];
            end = st[b + 1];
        } else if (ev) {
            g2h_aff p;
            g2h_load(p, sigs[ix[pos]]);
            pt_add_aff(R, R, p);
            pos++;
        }
    }
    if (pend) pt_add(T, T, S);
    if (!live) return;
    pt_mul_u64(R, R, (uint64_t)b);
    pt_add(T, T, R);
    g2h_store(out[id], T);
}
// pair members of the window sums: q[w] = W_w, p[w] = -[2^(8w)] G1 in pairing form
__global__ void k_msm_pairs(const g2_jac* vals, g2_jac* q, g1_pp* p) {
    const unsigned w = threadIdx.x;
    if (w >= B3_MSM_WINDOWS) return;
    q[w] = vals[w];
    g1_pp a;
    a.xz = G1_POW256_X[w]; a.ny = G1_POW256_Y[w]; a.z3 = FP_ONE; a.inf = 0;
    p[w] = a;
}

// pairwise tree level: out[i] = in[2i] + in[2i+1]   (LANE PAIRS: threads (2i, 2i+1) work on output i)
__global__ void __launch_bounds__(B3_TPB) k_g2_add_pairs(const g2_jac* in, size_t n, g2_jac* out) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    size_t m = (n + 1) / 2;
    if (i >= m) return;
    g2h_jac a;
    g2h_load(a, in[2 * i]);
    if (2 * i + 1 < n) {
        g2h_jac b;
        g2h_load(b, in[2 * i + 1]);
        pt_add(a, a, b);
    }
    g2h_store(out[i], a);
}

// ------------------------------------------------------------------------------------------------ normalisation
// Jacobian -> affine with MONTGOMERY'S TRICK (SURVEY.md a14): a thread normalises `per` consecutive points with ONE field
// inversion -- prefix products of the Z's, one binary-Euclid inversion (fp_inv: data-dependent control flow, the expensive
// and divergent part), then two multiplications per point to peel the individual inverses off.  The reference inverts once
// per point with a Fermat exponentiation (A/ecp.rs:362-379, A/ecp2.rs:203-218); the affine values are the same.
// G2: 1 / z = conj(z) / N(z), so the batch runs over the NORMS in Fp.
#define B3_NORM_MAX 16
__host__ __device__ __forceinline__ unsigned norm_per(size_t n) {          // points per thread: keep >= ~16 k threads
    size_t k = n / 16384;
    return k < 1 ? 1u : k > B3_NORM_MAX ? (unsigned)B3_NORM_MAX : (unsigned)k;
}
__global__ void __launch_bounds__(B3_TPB) k_g1_to_affine(const g1_jac* in, size_t n, g1_aff* out, unsigned per) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t first = t * per;
    if (first >= n) return;
    const unsigned cnt = (unsigned)(n - first < per ? n - first : per);
    fp pre[B3_NORM_MAX];
    fp acc = FP_ONE;
    for (unsigned j = 0; j < cnt; j++) {
        fp z = in[first + j].z;
        if (fp_is_zero(z)) z = FP_ONE;
        pre[j] = acc;
        fp_mul(acc, acc, z);
    }
    fp inv;
    fp_inv(inv, acc);
    for (unsigned j = cnt; j-- > 0;) {
        const g1_jac p = in[first + j];
        g1_aff a;
        if (fp_is_zero(p.z)) { a.x = FP_NIL; a.y = FP_NIL; a.inf = 1; }
        else {
            fp zi, zi2;
            fp_mul(zi, inv, pre[j]);
            fp_mul(inv, inv, p.z);
            fp_sqr(zi2, zi);
            fp_mul(a.x, p.x, zi2);
            fp_mul(zi2, zi2, zi);
            fp_mul(a.y, p.y, zi2);
            a.inf = 0;
        }
        out[first + j] = a;
    }
}
__global__ void __launch_bounds__(B3_TPB) k_g2_to_affine(const g2_jac* in, size_t n, g2_aff* out, unsigned per) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t first = t * per;
    if (first >= n) return;
    const unsigned cnt = (unsigned)(n - first < per ? n - first : per);
    fp pre[B3_NORM_MAX];
    fp acc = FP_ONE;
    for (unsigned j = 0; j < cnt; j++) {
        const fp2 z = in[first + j].z;
        fp nz, t1;
        fp_sqr(nz, z.c0);
        fp_sqr(t1, z.c1);
        fp_add(nz, nz, t1);                               // N(z) = 0 <=> z = 0 (-1 is not a square in Fp)
        if (fp_is_zero(nz)) nz = FP_ONE;
        pre[j] = acc;
        fp_mul(acc, acc, nz);
    }
    fp inv;
    fp_inv(inv, acc);
    for (unsigned j = cnt; j-- > 0;) {
        const g2_jac p = in[first + j];
        g2_aff a;
        if (fp2_is_zero(p.z)) { fp2_zero(a.x); fp2_zero(a.y); a.inf = 1; }
        else {
            fp nz, t1, ni;
            fp_sqr(nz, p.z.c0);
            fp_sqr(t1, p.z.c1);
            fp_add(nz, nz, t1);
            fp_mul(ni, inv, pre[j]);                      // 1 / N(z)
            fp_mul(inv, inv, nz);
            fp2 zi, zi2;
            fp_mul(zi.c0, p.z.c0, ni);
            fp_mul(t1, p.z.c1, ni);
            fp_neg(zi.c1, t1);                            // 1 / z = conj(z) / N(z)
            fp2_sqr(zi2, zi);
            fp2_mul(a.x, p.x, zi2);
            fp2_mul(zi2, zi2, zi);
            fp2_mul(a.y, p.y, zi2);
            a.inf = 0;
        }
        out[first + j] = a;
    }
}
__global__ void __launch_bounds__(B3_TPB) k_g1_aff_to_wire(const g1_aff* in, size_t n, uint8_t* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_aff a = in[i];
    g1_aff_to_wire(out + 96 * i, a);
}
__global__ void __launch_bounds__(B3_TPB) k_g2_aff_to_wire(const g2_aff* in, size_t n, uint8_t* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g2_aff a = in[i];
    g2_aff_to_wire(out + 192 * i, a);
}
// ------------------------------------------------------------------------------------------------ hash to G2
// Two threads per message.  Phase 1: each lane maps ONE of the two field elements to the curve (SSWU + 3-isogeny,
// single-thread Fp2 arithmetic: the square roots are chains of Fp operations).  Phase 2: the two points are
// redistributed into lane-pair form and the pair adds them and clears the cofactor together.
// The messages of a CTA (64 of them, contiguous in the blob) are STAGED: the CTA copies the byte range of its messages into
// shared memory with coalesced 16-byte loads (whole 16-byte words of the range; its ragged tail byte by byte) and every lane
// hashes from there.  Ranges that do not fit the stage (long messages) are read from global memory directly.
#define B3_H2C_STAGE_BYTES 4096
__global__ void __launch_bounds__(B3_TPB, B3_H2C_CTAS) k_hash_to_g2(const uint8_t* __restrict__ msgs, const uint32_t* __restrict__ off, size_t n,
                                                       const uint8_t* __restrict__ dst, uint32_t dst_len, g2_jac* out) {
    __shared__ uint4 stage[B3_H2C_STAGE_BYTES / 16];
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    const size_t m0 = ((size_t)blockIdx.x * blockDim.x) >> 1;                     // first message of this CTA (m0 < n for every CTA)
    const size_t m1 = m0 + (blockDim.x >> 1) < n ? m0 + (blockDim.x >> 1) : n;
    const uint32_t lo = off[m0], hi = off[m1];
    const uint32_t lo16 = lo & ~15u;
    const bool staged = hi - lo16 <= B3_H2C_STAGE_BYTES && (reinterpret_cast<uintptr_t>(msgs) & 15u) == 0;
    if (staged) {
        const uint32_t len = hi - lo16;
        for (uint32_t w = threadIdx.x; 16 * w < len; w += blockDim.x) {
            if (16 * w + 16 <= len) stage[w] = __ldg(reinterpret_cast<const uint4*>(msgs + lo16) + w);
            else
                for (uint32_t t = 16 * w; t < len; t++) reinterpret_cast<uint8_t*>(stage)[t] = msgs[lo16 + t];
        }
    }
    __syncthreads();
    if (i >= n) return;
    const bool odd = pair_odd();
    uint32_t b = off[i], e = off[i + 1];
    const uint8_t* msg = staged ? reinterpret_cast<const uint8_t*>(stage) + (b - lo16) : msgs + b;
    g2_jac q;
    {
        fp2 u0, u1, u;
        hash_to_field_fp2_x2(u0, u1, msg, e - b, dst, dst_len);
        fp2_select(u, odd, u1, u0);
        map_to_curve_g2(q, u);
    }
    // even lane holds Q0, odd lane holds Q1 -> (q0, q1) in lane-pair form
    g2h_jac q0, q1;
    const fp2* src[3] = {&q.x, &q.y, &q.z};
    fp2h* d0[3] = {&q0.x, &q0.y, &q0.z};
    fp2h* d1[3] = {&q1.x, &q1.y, &q1.z};
#pragma unroll
    for (int c = 0; c < 3; c++) {
        fp send, recv;
        fp_select(send, odd, src[c]->c0, src[c]->c1);      // even sends its c1 (for the odd lane), odd sends its c0
        pair_xchg(recv, send);
        fp_select(d0[c]->v, odd, recv, src[c]->c0);        // Q0: even keeps c0, odd receives Q0.c1
        fp_select(d1[c]->v, odd, src[c]->c1, recv);        // Q1: even receives Q1.c0, odd keeps c1
    }
    pt_add(q0, q0, q1);
    g2_clear_cofactor(q1, q0);
    g2h_store(out[i], q1);
}

// ------------------------------------------------------------------------------------------------ pairing
__global__ void __launch_bounds__(B3_TPB) k_g1_jac_to_pp(const g1_jac* in, size_t n, g1_pp* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_jac p = in[i];
    g1_pp r;
    g1_pp_from_jac(r, p);
    out[i] = r;
}
// P_j = [c_j] apk_j straight into pairing form
// zero_flag: set when a scalar is 0 -- the reference's draw rule never yields 0 (M/src/aggregates.rs:280-286), and a zero scalar
// would drop its set from the batch equation, so the call is rejected (B3_ERR_ARG)
__global__ void __launch_bounds__(B3_TPB) k_g1_mul_u64_pp(const g1_jac* in, const uint64_t* __restrict__ k, size_t n, g1_pp* out, int32_t* zero_flag) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g1_jac p = in[i], r;
    if (k[i] == 0) *zero_flag = 1;
    pt_mul_u64_w4(r, p, k[i]);
    g1_pp o;
    g1_pp_from_jac(o, r);
    out[i] = o;
}
// the same on LANE PAIRS (quad.cuh: fpd): threads (2i, 2i+1) work on set i, the paired products of the point formulas split
// over the two lanes
__global__ void __launch_bounds__(B3_TPB) k_g1_mul_u64_pp_d(const g1_jac* in, const uint64_t* __restrict__ k, size_t n, g1_pp* out, int32_t* zero_flag) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;
    g1d_jac p, r;
    g1d_load(p, in[i]);
    const uint64_t c = k[i];
    if (c == 0) *zero_flag = 1;
    pt_mul_u64_w4(r, p, c);
    // pairing form (X Z, -Y, Z^3): Z^2 and X Z as a pair, then Z^3
    fpd z2, xz, z3;
    f_mulsqr_par(xz, r.x, r.z, z2, r.z);
    f_mul(z3, z2, r.z);
    if (!pair_odd()) {
        g1_pp o;
        o.xz = xz.v;
        fp_neg(o.ny, r.y.v);
        o.z3 = z3.v;
        o.inf = fp_is_zero(r.z.v) ? 1u : 0u;
        out[i] = o;
    }
}
// constant pair member: -G1 generator
__global__ void k_set_neg_g1_pp(g1_pp* out) {
    g1_pp a;
    a.xz = G1_GEN_X; a.ny = G1_GEN_Y; a.z3 = FP_ONE; a.inf = 0;       // -( -y ) = y
    *out = a;
}
// parsed affine signature -> Jacobian pair member
__global__ void __launch_bounds__(B3_TPB) k_g2_aff_to_jac(const g2_aff* in, size_t n, g2_jac* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    g2_aff a = in[i];
    g2_jac j;
    pt_from_aff(j, a);
    out[i] = j;
}

// ---- split multi-Miller loop (pairing.cuh: "split Miller loop") ---------------------------------------------------
// 1. point chain of every pair -> unscaled lines, lines[(slot * n + pair) * 3 + {0,1,2}] = (u0, l3, u5)
//    LANE PAIRS: threads (2i, 2i+1) run the chain of pair i, each storing its half of every coefficient.
//    Pairs [first, first + count) of the n pairs of the product (different ranges may run on different streams).
__global__ void B3_LBH k_miller_lines(const g2_jac* __restrict__ q, size_t n, size_t first, size_t count,
                                                         fp2* __restrict__ lines, uint32_t* __restrict__ qinf) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= count) return;
    i += first;
    fp2h X, Y, Z;
    fp2h_load(X, q[i].x);
    fp2h_load(Y, q[i].y);
    fp2h_load(Z, q[i].z);
    const bool inf = fp2_is_zero(Z);
    if (!pair_odd()) qinf[i] = inf ? 1u : 0u;
    if (inf) return;                           // its lines are never read: the accumulate kernel skips the pair
    miller_pt_t<fp2h> t, Q;
    miller_start(t, X, Y, Z);
    Q = t;
    const uint64_t x = B3_X_ABS;
    int a = B3_MILLER_DBL_SLOTS;
    fp2h u0, l3, u5;
    for (int it = 0; it < B3_MILLER_DBL_SLOTS; it++) {
        miller_dbl_step_u(t, u0, l3, u5);
        fp2* o = lines + ((size_t)it * n + i) * 3;
        fp2h_store(o[0], u0); fp2h_store(o[1], l3); fp2h_store(o[2], u5);
        if ((x >> (62 - it)) & 1) {
            miller_add_step_u(t, u0, l3, u5, Q.x, Q.y, Q.z);
            o = lines + ((size_t)a * n + i) * 3;
            fp2h_store(o[0], u0); fp2h_store(o[1], l3); fp2h_store(o[2], u5);
            a++;
        }
    }
}
//    LANE QUADS (quad.cuh): threads 4i .. 4i+3 run the chain of pair i with the paired products of every step split over
//    the two lane pairs; the low pair stores u0 and l3, the high pair u5.
__global__ void B3_LBH k_miller_lines_q(const g2_jac* __restrict__ q, size_t n, size_t first, size_t count,
                                        fp2* __restrict__ lines, uint32_t* __restrict__ qinf) {
    size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 2;
    if (i >= count) return;
    i += first;
    fp2q X, Y, Z;
    fp2h_load(X, q[i].x);
    fp2h_load(Y, q[i].y);
    fp2h_load(Z, q[i].z);
    const bool inf = fp2_is_zero(Z);
    if ((threadIdx.x & 3u) == 0) qinf[i] = inf ? 1u : 0u;
    if (inf) return;                           // its lines are never read: the accumulate kernel skips the pair
    miller_pt_t<fp2q> t, Q;
    {                                          // homogeneous (X Z : Y : Z^3)
        fp2q z2;
        f_mulsqr_par(t.x, X, Z, z2, Z);
        t.y = Y;
        f_mul(t.z, z2, Z);
    }
    Q = t;
    const uint64_t x = B3_X_ABS;
    const bool hi = quad_hi();
    int a = B3_MILLER_DBL_SLOTS;
    fp2q u0, l3, u5;
    for (int it = 0; it < B3_MILLER_DBL_SLOTS; it++) {
        miller_dbl_step_u(t, u0, l3, u5);
        fp2* o = lines + ((size_t)it * n + i) * 3;
        if (hi) fp2h_store(o[2], u5);
        else { fp2h_store(o[0], u0); fp2h_store(o[1], l3); }
        if ((x >> (62 - it)) & 1) {
            miller_add_step_u(t, u0, l3, u5, Q.x, Q.y, Q.z);
            o = lines + ((size_t)a * n + i) * 3;
            if (hi) fp2h_store(o[2], u5);
            else { fp2h_store(o[0], u0); fp2h_store(o[1], l3); }
            a++;
        }
    }
}
// 2. slot accumulators, GROUP-COOPERATIVE: six lanes own one dense Fp12 accumulator, lane k holding the Fp2 coefficient of
//    w^k in registers (five groups per warp, lanes 30/31 idle; B3_ACC_GROUPS = 20 groups per CTA).  grid = (chunks,
//    B3_MILLER_SLOTS): group g of chunk c folds the lines of pairs [(c * 20 + g) K, +K) of its slot:
//      a. lane t scales one Fp coordinate of the line by its factor of P (times Z_P^3, an Fp factor) -> shared memory
//      b. the group derives the xi multiples and the sums X.c0 + X.c1 of the line operands in shared memory
//      c. lane k gathers the coefficients of w^(k+3) and w^(k+1) (and their c0 + c1) by warp shuffles and computes
//           r_k = l0 f_k + L3 f_{k-3} + L5 f_{k-5}      (L3 = l3 or xi l3, L5 = l5 or xi l5)
//         in Karatsuba form with THREE three-term dot products, one reduction each (fp_dot3_rs):
//           R0 = sum A.c0 B.c0,  R1 = sum A.c1 B.c1,  R2 = sum (A.c0 + A.c1)(B.c0 + B.c1);   re = R0 - R1,  im = R2 - R0 - R1
//         1764 multiply-accumulates per coefficient instead of 2040 for two six-term dot products (1.34 -> 1.24 ms).
//    The accumulator never leaves registers (the one-thread-per-accumulator version kept 2 x 576 B per thread in local
//    memory and thrashed L1: profiles/r1n_accum_full.txt).  The 20 group results are multiplied CTA-cooperatively;
//    partial[s * chunks + chunk] = product of the CTA's lines.
#define B3_ACC_GROUPS 20
// line operands of one group in shared memory: v[0..4] = X.c0, v[5..9] = X.c1, v[10..14] = X.c0 + X.c1 for X = l0, l3, xi l3, l5,
// xi l5, v[15] = 0 (operand of the lanes with nothing to derive), v[16], v[17] unused
struct acc_ops {
    fp v[18];
};
__global__ void __launch_bounds__(B3_TPB, 3) k_miller_accum(const fp2* __restrict__ lines, const uint32_t* __restrict__ qinf,
                                                            const g1_pp* __restrict__ p, size_t n, unsigned K, fp12* partial) {
    __shared__ acc_ops ops[B3_ACC_GROUPS];
    __shared__ fp12 tree[B3_ACC_GROUPS];
    __shared__ coop_ws ws;
    const unsigned slot = blockIdx.y, chunk = blockIdx.x, chunks = gridDim.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int gl = lane / 6, k = lane - 6 * gl;
    const bool live = gl < 5;
    const int g = warp * 5 + (live ? gl : 0);
    const int src3 = (6 * gl + (k + 3) % 6) & 31, src5 = (6 * gl + (k + 1) % 6) & 31;
    fp* const o = ops[g].v;
    // where lane k's scaled coordinate goes: (l0.c0, l0.c1, l3.c0, l3.c1, l5.c0, l5.c1) -> X slots 0, 1, 3
    fp* const mine = o + ((k & 1) ? 5 : 0) + ((k >> 1) == 2 ? 3 : (k >> 1));
    const int Z = 15, S0 = 16, S1 = 17;
    // branch-free derivation, lane k:  o[ksd] = o[ksx] - o[ksy];  t = o[kau] + o[kav] -> o[kad], o[kad2]
    //   k = 2, 3: xi l3 / xi l5 = (c0 - c1, c0 + c1), and c0 + c1 is also the sum of l3 / l5      k = 0: sum of l0
    //   k = 1, 4: sum of xi l3 / xi l5 = 2 c0 of l3 / l5                                            k = 5: nothing
    const int ksx = k == 2 ? 1 : k == 3 ? 3 : Z, ksy = k == 2 ? 6 : k == 3 ? 8 : Z, ksd = k == 2 ? 2 : k == 3 ? 4 : S0;
    const int kau = k == 0 ? 0 : k == 1 ? 1 : k == 2 ? 1 : k == 3 ? 3 : k == 4 ? 3 : Z;
    const int kav = k == 0 ? 5 : k == 1 ? 1 : k == 2 ? 6 : k == 3 ? 8 : k == 4 ? 3 : Z;
    const int kad = k == 0 ? 10 : k == 1 ? 12 : k == 2 ? 7 : k == 3 ? 9 : k == 4 ? 14 : S1;
    const int kad2 = k == 2 ? 11 : k == 3 ? 13 : S1;
    if (live && k == 0) o[Z] = FP_NIL;
    const int x3 = k >= 3 ? 1 : 2, x5 = k == 5 ? 3 : 4;
    const size_t first = ((size_t)chunk * B3_ACC_GROUPS + g) * K;
    fp a[6];                                               // a[0], a[1]: this lane's coefficient (c0, c1); a[2..5]: gathered
    a[0] = FP_NIL; a[1] = FP_NIL;
    bool have = false;
    for (unsigned it = 0; it < K; it++) {
        const size_t j = first + it;
        bool valid = live && j < n;
        if (valid) valid = !(qinf[j] || p[j].inf);
        if (valid) {
            fp v = reinterpret_cast<const fp*>(lines + ((size_t)slot * n + j) * 3)[k];
            const fp f = (k >> 1) == 0 ? p[j].ny : (k >> 1) == 1 ? p[j].z3 : p[j].xz;
            *mine = fp_mul_v(v, f);
        }
        __syncwarp();
        if (valid) {
            fp t;
            fp_sub(t, o[ksx], o[ksy]);
            if (k == 2 || k == 3) o[ksd] = t;              // predicated stores: lanes with nothing to derive write nothing
            fp_add(t, o[kau], o[kav]);
            if (k != 5) o[kad] = t;
            if (k == 2 || k == 3) o[kad2] = t;
        }
        __syncwarp();
        fp as0, as1, as2;                                  // c0 + c1 of this lane's coefficient and of the two gathered ones
        fp_add(as0, a[0], a[1]);
#pragma unroll
        for (int w = 0; w < 12; w++) {
            a[2].l[w] = __shfl_sync(0xffffffffu, a[0].l[w], src3);
            a[3].l[w] = __shfl_sync(0xffffffffu, a[1].l[w], src3);
            a[4].l[w] = __shfl_sync(0xffffffffu, a[0].l[w], src5);
            a[5].l[w] = __shfl_sync(0xffffffffu, a[1].l[w], src5);
            as1.l[w] = __shfl_sync(0xffffffffu, as0.l[w], src3);
            as2.l[w] = __shfl_sync(0xffffffffu, as0.l[w], src5);
        }
        if (valid) {
            if (have) {
                // r = sum_t A_t B_t over the three (coefficient, line operand) pairs, Karatsuba with three reductions:
                //   R2 = sum (A.c0 + A.c1)(B.c0 + B.c1), R0 = sum A.c0 B.c0, R1 = sum A.c1 B.c1;  re = R0 - R1, im = R2 - R0 - R1
                fp R0, R1, R2;
                R2 = fp_dot3_rs_v(as0, as1, as2, o + 10, o + 10 + x3, o + 10 + x5);
                R0 = fp_dot3_rs_v(a[0], a[2], a[4], o, o + x3, o + x5);
                R1 = fp_dot3_rs_v(a[1], a[3], a[5], o + 5, o + 5 + x3, o + 5 + x5);
                fp_sub(a[0], R0, R1);
                fp_sub(R2, R2, R0);
                fp_sub(a[1], R2, R1);
            } else {
                                          // first line: f = l0 + l3 w^3 + l5 w^5
                const int sl = k == 0 ? 0 : k == 3 ? 1 : 3;
                const bool nz = k == 0 || k == 3 || k == 5;
                fp_select(a[0], nz, o[sl], FP_NIL);
                fp_select(a[1], nz, o[5 + sl], FP_NIL);
                have = true;
            }
        }
        __syncwarp();
    }
    if (live) {
        if (!have) { fp_select(a[0], k == 0, FP_ONE, FP_NIL); a[1] = FP_NIL; }
        fp2& d = coop_coef(tree[g], k);
        d.c0 = a[0]; d.c1 = a[1];
    }
    __syncthreads();
    // groups that had pairs in range: at least one, at most all
    size_t left = n > (size_t)chunk * B3_ACC_GROUPS * K ? n - (size_t)chunk * B3_ACC_GROUPS * K : 0;
    unsigned used = (unsigned)((left + K - 1) / K);
    if (used > B3_ACC_GROUPS) used = B3_ACC_GROUPS;
    for (unsigned t = 1; t < used; t++) coop_fp12_mul(tree[0], tree[0], tree[t], ws);
    coop_copy_p(partial[(size_t)slot * chunks + chunk], tree[0], (int)threadIdx.x);
}
// 2b. one CTA per slot: slot value = product of that slot's per-chunk partials (only launched when chunks > 1)
__global__ void __launch_bounds__(B3_COOP_THREADS) k_miller_slots(const fp12* partial, unsigned chunks, fp12* slotvals) {
    __shared__ fp12 acc, tmp;
    __shared__ coop_ws ws;
    const unsigned s = blockIdx.x;
    COOP_PHASE(coop_copy_p(acc, partial[(size_t)s * chunks], tid));
    for (unsigned c = 1; c < chunks; c++) {
        COOP_PHASE(coop_copy_p(tmp, partial[(size_t)s * chunks + c], tid));
        coop_fp12_mul(acc, acc, tmp, ws);
    }
    coop_copy_p(slotvals[s], acc, (int)threadIdx.x);
}
// 3. one CTA: slot values = products of the per-chunk partials, then the closing sqr/mul chain -> *out
__global__ void __launch_bounds__(B3_COOP_THREADS) k_miller_chain(const fp12* partial, unsigned chunks, fp12* out) {
    __shared__ fp12 slots[B3_MILLER_SLOTS];
    __shared__ fp12 f, tmp;
    __shared__ coop_ws ws;
    for (unsigned s = 0; s < B3_MILLER_SLOTS; s++) {
        COOP_PHASE(coop_copy_p(slots[s], partial[(size_t)s * chunks], tid));
        for (unsigned c = 1; c < chunks; c++) {
            COOP_PHASE(coop_copy_p(tmp, partial[(size_t)s * chunks + c], tid));
            coop_fp12_mul(slots[s], slots[s], tmp, ws);
        }
    }
    coop_miller_chain(f, slots, ws);
    coop_copy_p(*out, f, (int)threadIdx.x);
}

// pairwise product tree level: out[i] = in[2i] * in[2i+1]
__global__ void __launch_bounds__(B3_TPB) k_fp12_mul_pairs(const fp12* in, size_t n, fp12* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    size_t m = (n + 1) / 2;
    if (i >= m) return;
    fp12 a = in[2 * i];
    if (2 * i + 1 < n) {
        fp12 b = in[2 * i + 1];
        fp12_mul(a, a, b);
    }
    out[i] = a;
}
__global__ void k_fp12_set_one(fp12* out) {
    fp12 a;
    fp12_one(a);
    *out = a;
}
// first failing index (or -1): min-reduction over ok[] == 0
__global__ void k_first_bad(const int32_t* ok, size_t n, long long index_base, long long* out) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (!ok[i]) atomicMin(out, index_base + (long long)i);
}
// Final exponentiation + is_unity + GT wire bytes: one CTA, cooperative Fp12 arithmetic (coop12.cuh)
__global__ void __launch_bounds__(B3_COOP_THREADS) k_final_exp(const fp12* in, uint8_t* gt_wire, int32_t* is_one) {
    __shared__ coop_fexp_ws s;
    COOP_PHASE(coop_copy_p(s.m, *in, tid));
    coop_final_exp(s);
    const int tid = (int)threadIdx.x;
    if (tid < 12) {                                   // wire order w^0, w^3, w^1, w^4, w^2, w^5, each (re, im)
        const int order[6] = {0, 3, 1, 4, 2, 5};
        const fp2& c = coop_coef(s.rr, order[tid >> 1]);
        fp t;
        fp_from_mont(t, (tid & 1) ? c.c1 : c.c0);
        fp_raw_to_be(gt_wire + 48 * tid, t);
    }
    if (tid == 0) *is_one = fp12_is_one(s.rr) ? 1 : 0;
}

// ---- batched PER-ITEM verification (b3_verify_batch, b3_verify_multiple_locate): one CTA per item -------------------
// Item i owns two pairs: (sig_i, -G1), whose lines are pair first0 + i of the np0-pair table lines0 (qinf0), and
// (H(msg_i), key_i), pair first1 + i of the np1-pair table lines1 (b3_verify_batch passes its one 2n-pair table twice, with
// first0 = 0 and first1 = n).  The CTA folds the 2 x 68 lines into its own accumulator (sparse cooperative products), runs
// its own final exponentiation and writes the item's accept bit, status (nullable) and GT bytes (nullable) -- the shape of
// `ate2` + `fexp` (A/pair.rs:313-541) per item.
// Items the reference rejects before any pairing skip the arithmetic altogether, by key_rule:
//   B3_KEY_INF_PAIR    bad encoding or subgroup check (M/src/signature.rs:29-31); an infinite key contributes 1
//   B3_KEY_INF_REJECT  ... and an empty or infinite aggregate key (M/src/aggregates.rs:179-198,229-236)
//   B3_KEY_BATCH       the rule of one set of verify_multiple (M/src/aggregates.rs:261-316): an empty key list
//                      (B3_ERR_AGGREGATE_EMPTY_POINTS) or an infinite aggregate key rejects nothing, its pair contributes 1
#define B3_KEY_INF_PAIR 0
#define B3_KEY_INF_REJECT 1
#define B3_KEY_BATCH 2
__device__ __forceinline__ int item_code(const int32_t* st_sig, const int32_t* st_key, size_t i, int key_rule) {
    const int kc = st_key[i];
    return st_sig[i] ? st_sig[i] : (key_rule == B3_KEY_BATCH && kc == B3_ERR_AGGREGATE_EMPTY_POINTS_D) ? 0 : kc;
}
__global__ void __launch_bounds__(B3_COOP_THREADS) k_items_finish(const fp2* __restrict__ lines0, const uint32_t* __restrict__ qinf0, size_t np0,
                                                                  size_t first0, const fp2* __restrict__ lines1, const uint32_t* __restrict__ qinf1,
                                                                  size_t np1, size_t first1, const g1_pp* __restrict__ keys, const int32_t* st_sig,
                                                                  const int32_t* st_key, const int32_t* sig_ok, int key_rule,
                                                                  int32_t* accept, int32_t* status, uint8_t* gt_wire) {
    __shared__ coop_fexp_ws s;
    __shared__ fp12 line;
    __shared__ coop_item_pair pr[2];
    const size_t i = blockIdx.x;
    const int code = item_code(st_sig, st_key, i, key_rule);
    const bool rejected = code != 0 || !sig_ok[i] || (key_rule == B3_KEY_INF_REJECT && keys[i].inf);
    if (rejected) {                                    // uniform over the CTA
        if (threadIdx.x == 0) { accept[i] = 0; if (status) status[i] = code; }
        if (gt_wire) for (int b = threadIdx.x; b < 576; b += blockDim.x) gt_wire[576 * i + b] = 0;
        return;
    }
    if (threadIdx.x == 0) {
        pr[0].idx = first0 + i; pr[0].ny = G1_GEN_Y; pr[0].z3 = FP_ONE; pr[0].xz = G1_GEN_X;          // -G1: -(-y) = y
        pr[0].valid = qinf0[first0 + i] ? 0 : 1;
        pr[0].lines = lines0; pr[0].np = np0;
        const g1_pp k = keys[i];
        pr[1].idx = first1 + i; pr[1].ny = k.ny; pr[1].z3 = k.z3; pr[1].xz = k.xz;
        pr[1].valid = (qinf1[first1 + i] || k.inf) ? 0 : 1;
        pr[1].lines = lines1; pr[1].np = np1;
    }
    __syncthreads();
    coop_item_miller(s.m, line, s.ws, nullptr, 0, pr, 2);
    coop_final_exp(s);
    const int tid = (int)threadIdx.x;
    if (gt_wire && tid < 12) {                        // wire order w^0, w^3, w^1, w^4, w^2, w^5, each (re, im)
        const int order[6] = {0, 3, 1, 4, 2, 5};
        const fp2& c = coop_coef(s.rr, order[tid >> 1]);
        fp t;
        fp_from_mont(t, (tid & 1) ? c.c1 : c.c0);
        fp_raw_to_be(gt_wire + 576 * i + 48 * tid, t);
    }
    if (tid == 0) { accept[i] = fp12_is_one(s.rr) ? 1 : 0; if (status) status[i] = 0; }
}

// The same work with a LANE PAIR per item (large batches): a CTA per item keeps at most 2 x 148 items in flight, a lane pair per item
// keeps every item of the batch in flight.  The Fp6 / Fp12 tower and the final exponentiation are templates over the
// Fp2 representation (tower.cuh, pairing.cuh), so the same chain runs with every Fp2 value split over two lanes (fp2h.cuh):
// half the latency of the thread-per-item kernel and twice the threads.  Sparse products use the Karatsuba form
// (fp12_mul_by_line: 14 Fp2 products, each 444 multiply-accumulates per lane).
#define B3_ITEMS_PAIR_TPB 64
__device__ __noinline__ void item_fold_line_p(fp12_t<fp2h>& f, bool& have, const fp2* __restrict__ src, const fp& ny, const fp& z3, const fp& xz) {
    fp2h l0, l3, l5;
    fp2h_load(l0, src[0]); fp2h_load(l3, src[1]); fp2h_load(l5, src[2]);
    fp2_mul_fp(l0, l0, ny);
    fp2_mul_fp(l3, l3, z3);
    fp2_mul_fp(l5, l5, xz);
    if (have) fp12_mul_by_line(f, l0, l3, l5);
    else { fp12_from_line(f, l0, l3, l5); have = true; }
}
__global__ void __launch_bounds__(B3_ITEMS_PAIR_TPB) k_items_finish_p(const fp2* __restrict__ lines0, const uint32_t* __restrict__ qinf0,
                                                                       size_t np0, size_t first0, const fp2* __restrict__ lines1,
                                                                       const uint32_t* __restrict__ qinf1, size_t np1, size_t first1,
                                                                       const g1_pp* __restrict__ keys, size_t n, const int32_t* st_sig,
                                                                       const int32_t* st_key, const int32_t* sig_ok, int key_rule,
                                                                       int32_t* accept, int32_t* status, uint8_t* gt_wire) {
    const size_t i = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 1;
    if (i >= n) return;                                // both lanes of a pair leave together
    const bool odd = pair_odd();
    const int code = item_code(st_sig, st_key, i, key_rule);
    const g1_pp key = keys[i];
    if (code != 0 || !sig_ok[i] || (key_rule == B3_KEY_INF_REJECT && key.inf)) {
        if (!odd) { accept[i] = 0; if (status) status[i] = code; }
        if (gt_wire) for (int b = odd ? 288 : 0; b < (odd ? 576 : 288); b++) gt_wire[576 * i + b] = 0;
        return;
    }
    const bool valid0 = !qinf0[first0 + i], valid1 = !(qinf1[first1 + i] || key.inf);
    const fp gy = G1_GEN_Y, one = FP_ONE, gx = G1_GEN_X;           // pair 0 = (sig_i, -G1): -(-y) = y
    fp12_t<fp2h> f, g;
    bool have = false;
    const uint64_t x = B3_X_ABS;
    int a = B3_MILLER_DBL_SLOTS;
#pragma unroll 1
    for (int it = 0; it < B3_MILLER_DBL_SLOTS; it++) {
        if (have) fp12_sqr(f, f);
        const bool add = (x >> (62 - it)) & 1;
#pragma unroll 1
        for (int s = 0; s < (add ? 2 : 1); s++) {
            const size_t slot = s == 0 ? (size_t)it : (size_t)a;
            if (valid0) item_fold_line_p(f, have, lines0 + (slot * np0 + first0 + i) * 3, gy, one, gx);
            if (valid1) item_fold_line_p(f, have, lines1 + (slot * np1 + first1 + i) * 3, key.ny, key.z3, key.xz);
        }
        if (add) a++;
    }
    if (!have) fp12_one(f);
    fp12_conj(f, f);
    final_exp(g, f);
    const bool is_one = fp12_is_one(g);
    if (gt_wire) {                                     // wire order w^0, w^3, w^1, w^4, w^2, w^5, each (re, im): this lane writes its half
        const int order[6] = {0, 3, 1, 4, 2, 5};
        for (int k = 0; k < 6; k++) {
            fp t;
            fp_from_mont(t, fp12_coef(g, order[k]).v);
            fp_raw_to_be(gt_wire + 576 * i + 96 * k + (odd ? 48 : 0), t);
        }
    }
    if (!odd) { accept[i] = is_one ? 1 : 0; if (status) status[i] = 0; }
}

// ------------------------------------------------------------------------------------------------ roofline microbenchmarks
// Pure integer-multiply issue-rate probes: `iters` rounds of 8 independent chains per thread.
__global__ void __launch_bounds__(256) k_imad_peak(uint32_t* out, int iters, uint32_t seed) {
    uint32_t a0 = seed + threadIdx.x, a1 = a0 * 3 + 1, a2 = a0 * 5 + 2, a3 = a0 * 7 + 3;
    uint32_t a4 = a0 * 11 + 4, a5 = a0 * 13 + 5, a6 = a0 * 17 + 6, a7 = a0 * 19 + 7;
    uint32_t m = seed | 1u, c = seed ^ 0x9e3779b9u;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            a0 = a0 * m + c; a1 = a1 * m + c; a2 = a2 * m + c; a3 = a3 * m + c;
            a4 = a4 * m + c; a5 = a5 * m + c; a6 = a6 * m + c; a7 = a7 * m + c;
        }
    }
    out[blockIdx.x * blockDim.x + threadIdx.x] = a0 ^ a1 ^ a2 ^ a3 ^ a4 ^ a5 ^ a6 ^ a7;
}
__global__ void __launch_bounds__(256) k_imad_wide_peak(uint32_t* out, int iters, uint32_t seed) {
    uint32_t lo[8], hi[8];
#pragma unroll
    for (int k = 0; k < 8; k++) { lo[k] = seed + threadIdx.x * (k + 1); hi[k] = seed ^ (k * 77u); }
    uint32_t m = seed | 1u, x = threadIdx.x | 3u;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 4; u++) {
            // two independent 4-pair carry chains, the shape of b3_mad_row
            mad_wide_cc(lo[0], hi[0], x, m); madc_wide_cc(lo[1], hi[1], x, m); madc_wide_cc(lo[2], hi[2], x, m); madc_wide_cc(lo[3], hi[3], x, m);
            mad_wide_cc(lo[4], hi[4], x, m); madc_wide_cc(lo[5], hi[5], x, m); madc_wide_cc(lo[6], hi[6], x, m); madc_wide_cc(lo[7], hi[7], x, m);
        }
    }
    uint32_t r = 0;
#pragma unroll
    for (int k = 0; k < 8; k++) r ^= lo[k] ^ hi[k];
    out[blockIdx.x * blockDim.x + threadIdx.x] = r;
}
