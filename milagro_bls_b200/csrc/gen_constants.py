#!/usr/bin/env python3
"""Generates constants.cuh (Montgomery form, R = 2^384, 12 x 32-bit little-endian limbs).

Stand-alone: derives every constant from the BLS12-381 parameters (p, r, x, generators) and the
RFC 9380 section 8.8.2 / E.3 suite constants.  Run by hand when the set of constants changes:
    python milagro_bls_b200/csrc/gen_constants.py
The values are cross-checked against the oracle by tests/test_constants.py.
"""
import pathlib

p = 0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaaab
r = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
X_ABS = 0xd201000000010000
R = 1 << 384
G1X = 0x17f1d3a73197d7942695638c4fa9ac0fc3688c4f9774b905a14e3a3f171bac586c55e83ff97a1aeffb3af00adb22c6bb
G1Y = 0x08b3f481e3aaa0f1a09e30ed741d8ae4fcf5e095d5d00af600db18cb2c04b3edd03cc744a2888ae40caa232946c5e7e1

ISO3_XNUM = [
    (0x5c759507e8e333ebb5b7a9a47d7ed8532c52d39fd3a042a88b58423c50ae15d5c2638e343d9c71c6238aaaaaaaa97d6,
     0x5c759507e8e333ebb5b7a9a47d7ed8532c52d39fd3a042a88b58423c50ae15d5c2638e343d9c71c6238aaaaaaaa97d6),
    (0x0,
     0x11560bf17baa99bc32126fced787c88f984f87adf7ae0c7f9a208c6b4f20a4181472aaa9cb8d555526a9ffffffffc71a),
    (0x11560bf17baa99bc32126fced787c88f984f87adf7ae0c7f9a208c6b4f20a4181472aaa9cb8d555526a9ffffffffc71e,
     0x8ab05f8bdd54cde190937e76bc3e447cc27c3d6fbd7063fcd104635a790520c0a395554e5c6aaaa9354ffffffffe38d),
    (0x171d6541fa38ccfaed6dea691f5fb614cb14b4e7f4e810aa22d6108f142b85757098e38d0f671c7188e2aaaaaaaa5ed1,
     0x0),
]
ISO3_XDEN = [
    (0x0,
     0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaa63),
    (0xc,
     0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaa9f),
    (0x1, 0x0),
]
ISO3_YNUM = [
    (0x1530477c7ab4113b59a4c18b076d11930f7da5d4a07f649bf54439d87d27e500fc8c25ebf8c92f6812cfc71c71c6d706,
     0x1530477c7ab4113b59a4c18b076d11930f7da5d4a07f649bf54439d87d27e500fc8c25ebf8c92f6812cfc71c71c6d706),
    (0x0,
     0x5c759507e8e333ebb5b7a9a47d7ed8532c52d39fd3a042a88b58423c50ae15d5c2638e343d9c71c6238aaaaaaaa97be),
    (0x11560bf17baa99bc32126fced787c88f984f87adf7ae0c7f9a208c6b4f20a4181472aaa9cb8d555526a9ffffffffc71c,
     0x8ab05f8bdd54cde190937e76bc3e447cc27c3d6fbd7063fcd104635a790520c0a395554e5c6aaaa9354ffffffffe38f),
    (0x124c9ad43b6cf79bfbf7043de3811ad0761b0f37a1e26286b0e977c69aa274524e79097a56dc4bd9e1b371c71c718b10,
     0x0),
]
ISO3_YDEN = [
    (0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffa8fb,
     0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffa8fb),
    (0x0,
     0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffa9d3),
    (0x12,
     0x1a0111ea397fe69a4b1ba7b6434bacd764774b84f38512bf6730d2a0f6b0f6241eabfffeb153ffffb9feffffffffaa99),
    (0x1, 0x0),
]


# ---- tiny Fp2 helpers --------------------------------------------------------------------------
def f2mul(a, b):
    return ((a[0] * b[0] - a[1] * b[1]) % p, (a[0] * b[1] + a[1] * b[0]) % p)


def f2pow(a, e):
    out = (1, 0)
    while e:
        if e & 1:
            out = f2mul(out, a)
        a = f2mul(a, a)
        e >>= 1
    return out


def f2inv(a):
    n = pow(a[0] * a[0] + a[1] * a[1], -1, p)
    return (a[0] * n % p, -a[1] * n % p)


def f2conj(a):
    return (a[0], -a[1] % p)


XI = (1, 1)
FROB = f2pow(XI, (p - 1) // 6)                 # w^p = FROB * w    (w^6 = xi)
GAMMA1 = [f2pow(FROB, k) for k in range(6)]   # (w^k)^p   = GAMMA1[k] * w^k  (applied after conj)
GAMMA2 = [f2mul(f2conj(g), g) for g in GAMMA1]                       # p^2 : in Fp
GAMMA3 = [f2mul(f2conj(GAMMA2[k]), GAMMA1[k]) for k in range(6)]     # p^3
for g in GAMMA2:
    assert g[1] == 0
PSI_X = f2inv(FROB)                            # untwist-Frobenius-twist constant of the M-type twist
PSI_CX = f2mul(PSI_X, PSI_X)
PSI_CY = f2mul(PSI_CX, PSI_X)
PSI2_CX = f2mul(f2conj(PSI_CX), PSI_CX)
PSI2_CY = f2mul(f2conj(PSI_CY), PSI_CY)
assert PSI2_CX[1] == 0 and PSI2_CY[1] == 0

# cube root of unity beta with phi(x,y) = (beta x, y) acting as [-x^2] on G1
def g1_add(P, Q):
    if P is None:
        return Q
    if Q is None:
        return P
    if P[0] == Q[0]:
        if (P[1] + Q[1]) % p == 0:
            return None
        lam = 3 * P[0] * P[0] * pow(2 * P[1], -1, p) % p
    else:
        lam = (Q[1] - P[1]) * pow(Q[0] - P[0], -1, p) % p
    x3 = (lam * lam - P[0] - Q[0]) % p
    return (x3, (lam * (P[0] - x3) - P[1]) % p)


def g1_mul(P, e):
    Rr = None
    for bit in bin(e)[2:]:
        Rr = g1_add(Rr, Rr)
        if bit == "1":
            Rr = g1_add(Rr, P)
    return Rr


_b = pow(2, (p - 1) // 3, p)
assert _b != 1 and pow(_b, 3, p) == 1
_target = g1_mul((G1X, G1Y), (-X_ABS * X_ABS) % r)
BETA = None
for cand in (_b, _b * _b % p):
    if (cand * G1X % p, G1Y) == _target:
        BETA = cand
assert BETA is not None

SQRT_M5 = pow(-5 % p, (p + 1) // 4, p)
assert SQRT_M5 * SQRT_M5 % p == (-5) % p
SSWU_A = (0, 240)
SSWU_B = (1012, 1012)
SSWU_Z = ((-2) % p, (-1) % p)
assert SSWU_Z[0] ** 2 + SSWU_Z[1] ** 2 == 5 + (SSWU_Z[0] ** 2 + SSWU_Z[1] ** 2 - 5) and \
    (SSWU_Z[0] ** 2 + SSWU_Z[1] ** 2) % p == 5
SSWU_ZA = f2mul(SSWU_Z, SSWU_A)

G2X = (0x024aa2b2f08f0a91260805272dc51051c6e47ad4fa403b02b4510b647ae3d1770bac0326a805bbefd48056c8c121bdb8,
       0x13e02b6052719f607dacd3a088274f65596bd0d09920b61ab5da61bbdc7f5049334cf11213945d57e5ac7d055d042b7e)
G2Y = (0x0ce5d527727d6e118cc9cdc6da2e351aadfd9baa8cbdd3a76d429a695160d12c923ac9cc3baca289e193548608b82801,
       0x0606c4a02ea734cc32acd2b02bc28b99cb3e287e85a763af267492ab572e99ab3f370d275cec1da1aaa9075ff05f79be)


# ---- emit --------------------------------------------------------------------------------------
def limbs(v, n=12):
    return "{" + ", ".join("0x%08xu" % ((v >> (32 * i)) & 0xFFFFFFFF) for i in range(n)) + "}"


def mont(v):
    return v * R % p


def fp_c(name, v, raw=False):
    return "B3_CONST fp %s = {%s};" % (name, limbs(v if raw else mont(v)))


def fp2_c(name, v):
    return "B3_CONST fp2 %s = {{%s}, {%s}};" % (name, limbs(mont(v[0])), limbs(mont(v[1])))


def fp2_arr(name, vs):
    body = ",\n    ".join("{{%s}, {%s}}" % (limbs(mont(v[0])), limbs(mont(v[1]))) for v in vs)
    return "B3_CONST fp2 %s[%d] = {\n    %s};" % (name, len(vs), body)


def fp_arr(name, vs):
    body = ",\n    ".join("{%s}" % limbs(mont(v)) for v in vs)
    return "B3_CONST fp %s[%d] = {\n    %s};" % (name, len(vs), body)


out = ["// GENERATED by gen_constants.py -- do not edit.  Montgomery form, R = 2^384, little-endian u32 limbs.",
       "#pragma once", ""]
out.append(fp_c("FP_P", p, raw=True))
out.append(fp_c("FP_2P", 2 * p, raw=True))
out.append(fp_c("FP_NIL", 0, raw=True))
out.append(fp_c("FP_ONE", 1))
out.append(fp_c("FP_RAW_ONE", 1, raw=True))
out.append(fp_c("FP_M_ONE", p - 1))
out.append(fp_c("FP_R2", R % p))                 # mont(R)   = R^2 mod p
out.append(fp_c("FP_R3", R * R % p))             # mont(R^2) = R^3 mod p
out.append("#define FP_PINV32 0x%08xu   /* -p^-1 mod 2^32 */" % ((-pow(p, -1, 1 << 32)) % (1 << 32)))
out.append(fp_c("FP_EXP_INV", p - 2, raw=True))
out.append(fp_c("FP_EXP_SQRT_G", (p - 3) // 4, raw=True))
out.append(fp_c("FP_BETA", BETA))
out.append(fp_c("FP_SQRT_M5", SQRT_M5))
out.append(fp_c("G1_GEN_X", G1X))
out.append(fp_c("G1_GEN_Y", G1Y))
out.append(fp_c("G1_GEN_NEG_Y", (-G1Y) % p))
# [2^(8w)] G1, w = 0..7: G1 members of the per-window pairs of the bucket-method sum (kernels.cuh, k_msm_*)
_pow = [g1_mul((G1X, G1Y), 1 << (8 * w)) for w in range(8)]
out.append(fp_arr("G1_POW256_X", [P[0] for P in _pow]))
out.append(fp_arr("G1_POW256_Y", [P[1] for P in _pow]))
out.append(fp2_c("G2_GEN_X", G2X))
out.append(fp2_c("G2_GEN_Y", G2Y))
out.append(fp2_arr("FROB_GAMMA1", GAMMA1))
out.append(fp_arr("FROB_GAMMA2", [g[0] for g in GAMMA2]))
out.append(fp2_arr("FROB_GAMMA3", GAMMA3))
out.append(fp2_c("PSI_CX", PSI_CX))
out.append(fp2_c("PSI_CY", PSI_CY))
out.append(fp_c("PSI2_CX", PSI2_CX[0]))
out.append(fp_c("PSI2_CY", PSI2_CY[0]))
out.append(fp2_c("SSWU_A", SSWU_A))
out.append(fp2_c("SSWU_B", SSWU_B))
out.append(fp2_c("SSWU_Z", SSWU_Z))
out.append(fp2_c("SSWU_ZA", SSWU_ZA))
out.append(fp2_arr("ISO3_XNUM", ISO3_XNUM))
out.append(fp2_arr("ISO3_XDEN", ISO3_XDEN))
out.append(fp2_arr("ISO3_YNUM", ISO3_YNUM))
out.append(fp2_arr("ISO3_YDEN", ISO3_YDEN))
out.append("#define B3_X_ABS 0xd201000000010000ull   /* |x|, the curve parameter is -|x| */")
out.append("")
pathlib.Path(__file__).with_name("constants.cuh").write_text("\n".join(out))
print("constants.cuh written; beta = %x" % BETA)
