"""The field layer keeps device values in [0, 2p), not necessarily canonical (milagro_bls_b200/csrc/fp.cuh).  Every Fp
primitive, compiled for the host (tests/hostsim/hostsim_relaxed.cpp), is fed adversarial operands in [p, 2p) next to
canonical ones; each result must stay below 2p (canonical where the primitive promises it) and equal the oracle's value
mod p."""
import ctypes
import itertools
import os
import random
import subprocess

import pytest

from oracle import bls_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsim", "hostsim_relaxed.cpp")

p = O.p
R = 1 << 384
RINV = pow(R, -1, p)
rnd = random.Random(2024)

# Montgomery residues as stored on the device: canonical edges, their non-canonical twins v + p, and random values
CANON = [0, 1, 2, p - 1, p - 2, (p - 1) // 2, (p + 1) // 2, R % p, (R * R) % p]
ADVERSARIAL = [p, p + 1, 2 * p - 1, 2 * p - 2, p + (p - 1) // 2, p + R % p, p + (R * R) % p]
VALUES = CANON + ADVERSARIAL + [rnd.randrange(p) for _ in range(8)] + [p + rnd.randrange(p) for _ in range(16)]


@pytest.fixture(scope="module")
def hs(tmp_path_factory):
    lib = str(tmp_path_factory.mktemp("hostsim") / "libhostsim_relaxed.so")
    subprocess.check_call(["g++", "-O2", "-std=c++17", "-x", "c++", "-shared", "-fPIC", "-o", lib, SRC])
    h = ctypes.CDLL(lib)
    h.hs_fp_raw.argtypes = [ctypes.c_int] + [ctypes.c_char_p] * 5
    h.hs_fp_dot6_raw.argtypes = [ctypes.c_char_p] * 3
    return h


def le(v):
    return v.to_bytes(48, "little")


def op(hs, code, a, b=0, c=0, d=0):
    out = ctypes.create_string_buffer(48)
    hs.hs_fp_raw(code, le(a), le(b), le(c), le(d), out)
    return out.raw


def rop(hs, code, *args):
    return int.from_bytes(op(hs, code, *args), "little")


def val(x):
    """field element a Montgomery residue stands for"""
    return x * RINV % p


def check(r, want):
    assert r < 2 * p, hex(r)
    assert val(r) == want % p


def pairs():
    return list(itertools.product(VALUES, VALUES))[::3] + [(a, b) for a in ADVERSARIAL for b in ADVERSARIAL]


def test_products(hs):
    for a, b in pairs():
        check(rop(hs, 0, a, b), val(a) * val(b))
        check(rop(hs, 2, a, b, b, a), 2 * val(a) * val(b))
        check(rop(hs, 2, a, a, b, b), val(a) ** 2 + val(b) ** 2)
    for a in VALUES:
        check(rop(hs, 1, a), val(a) ** 2)


def test_add_sub_neg_dbl_half(hs):
    for a, b in pairs():
        check(rop(hs, 3, a, b), val(a) + val(b))
        check(rop(hs, 4, a, b), val(a) - val(b))
    for a in VALUES:
        check(rop(hs, 5, a), -val(a))
        check(rop(hs, 6, a), 2 * val(a))
        check(rop(hs, 7, a), val(a) * pow(2, -1, p))


def test_canonical_forms(hs):
    for a in VALUES:
        assert rop(hs, 8, a) == a % p
        assert rop(hs, 9, a) == val(a)
        assert op(hs, 11, a) == (a % p).to_bytes(48, "big")
        assert op(hs, 12, a)[0] == (a % p == 0)
        r = rop(hs, 10, a)
        if a % p == 0:
            assert r == 0
        else:
            check(r, pow(val(a), -1, p))
    for a, b in pairs():
        assert op(hs, 13, a, b)[0] == (a % p == b % p)


def test_unreduced_product_operands(hs):
    """a + b < 4p and 2p - a in (0, 2p] are valid product operands: the result is below 2p again"""
    for (a, b), c in zip(pairs(), itertools.cycle(VALUES[::-1])):
        check(rop(hs, 14, a, b, c), (val(a) + val(b)) * val(c))
        check(rop(hs, 15, a, b, c, c), val(c) ** 2 - val(a) * val(b))
    m = 2 * p - 1
    check(rop(hs, 14, m, m, m), 2 * val(m) ** 2)
    check(rop(hs, 15, 0, m, m, m), val(m) ** 2)
    assert rop(hs, 16, 0) == 2 * p
    for a in VALUES:
        n = rop(hs, 16, a)
        assert 0 < n <= 2 * p and val(n) == -val(a) % p


def test_dot6(hs):
    for k in range(40):
        pool = ADVERSARIAL if k < 20 else VALUES
        a = [rnd.choice(pool) for _ in range(6)]
        b = [rnd.choice(pool) for _ in range(6)]
        if k == 0:
            a = b = [2 * p - 1] * 6
        out = ctypes.create_string_buffer(48)
        hs.hs_fp_dot6_raw(b"".join(map(le, a)), b"".join(map(le, b)), out)
        check(int.from_bytes(out.raw, "little"), sum(val(x) * val(y) for x, y in zip(a, b)))
