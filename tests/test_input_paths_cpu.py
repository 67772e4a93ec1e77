"""CPU companions of tests/test_gpu_input_paths.py.

(a) The GPU file builds its shapes from Python restatements of three selection rules (the hash_to_G2 stage, the lanes per set
    of the aggregation kernels, the points per inversion of the normalisation).  If a threshold moves in the sources, the
    shapes silently stop reaching the path they were made for; this test fails instead and names the constant to update.
(b) The host replay of hash_to_field (the device code compiled for the host, tests/hostsim) against the Python oracle over the
    message and DST lengths where SHA-256 block boundaries move."""
import ctypes
import importlib.util
import os
import re

import pytest

from oracle import bls_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "..", "milagro_bls_b200", "csrc")


def _load(name):
    spec = importlib.util.spec_from_file_location(name, os.path.join(HERE, name + ".py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


R = _load("test_gpu_input_paths")
hs = _load("test_hostsim").hs                     # the host replay library (module-scoped fixture)


def _src(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _one(pattern, text, what):
    m = re.findall(pattern, text)
    assert len(m) == 1, f"{what}: the source no longer matches {pattern!r}; update the rules of tests/test_gpu_input_paths.py"
    return m[0]


def test_selection_rule_constants_match_sources():
    kern, capi = _src("kernels.cuh"), _src("capi.cu")
    assert int(_one(r"#define B3_TPB (\d+)", kern, "B3_TPB")) == R.B3_TPB
    assert int(_one(r"#define B3_H2C_STAGE_BYTES (\d+)", kern, "B3_H2C_STAGE_BYTES")) == R.H2C_STAGE_BYTES
    # k_hash_to_g2: two threads per message, B3_TPB threads per CTA, stage used only from a 16-byte aligned blob
    assert len(re.findall(r"LAUNCH_ON\(strm, k_hash_to_g2, nblk\(2 \* n\), B3_TPB,", capi)) == 2            # Jacobian and affine forms
    assert len(re.findall(r"k_hash_to_g2\b", capi)) == 2
    _one(r"const size_t m1 = m0 \+ \(blockDim\.x >> 1\) < n", kern, "messages per CTA")
    _one(r"const bool staged = hi - lo16 <= B3_H2C_STAGE_BYTES && \(reinterpret_cast<uintptr_t>\(msgs\) & 15u\) == 0;", kern, "stage rule")
    _one(r"const uint32_t lo16 = lo & ~15u;", kern, "stage start")
    # launch_agg: G = 4 from g4_min sets or <= 8 keys per set, 8 from 2048 sets or <= 32, else 32
    assert int(_one(r"static const size_t kAggG4Min = (\d+);", capi, "kAggG4Min")) == R.AGG_G4_MIN_G1
    _one(r"if \(n_sets >= g4_min \|\| avg <= 8\) LAUNCH_ON\(strm, kern_of\(std::integral_constant<int, 4>\(\)\)", capi, "G = 4 rule")
    _one(r"else if \(n_sets >= 2048 \|\| avg <= 32\) LAUNCH_ON\(strm, kern_of\(std::integral_constant<int, 8>\(\)\)", capi, "G = 8 rule")
    _one(r"else LAUNCH_ON\(strm, kern_of\(std::integral_constant<int, 32>\(\)\)", capi, "G = 32 rule")
    _one(r"const size_t avg = total_keys / n_sets;", capi, "average set size")
    assert len(re.findall(r"launch_agg\(ctx, strm, n_sets, total_keys, kAggG4Min,", capi)) == 2           # G1 bytes and table
    assert int(_one(r"launch_agg\(ctx, ctx->stream, n_sets, total, (\d+), \[\]\(auto g\) \{ return k_g2_aggregate", capi,
                    "G2 g4_min")) == R.AGG_G4_MIN_G2
    # norm_per: clamp(n / 16384, 1, B3_NORM_MAX)
    assert int(_one(r"#define B3_NORM_MAX (\d+)", kern, "B3_NORM_MAX")) == R.NORM_MAX
    assert int(_one(r"size_t k = n / (\d+);", kern, "norm_per divisor")) == R.NORM_POINTS_PER_THREAD
    _one(r"return k < 1 \? 1u : k > B3_NORM_MAX \? \(unsigned\)B3_NORM_MAX : \(unsigned\)k;", kern, "norm_per clamp")


def test_selection_rules_restated():
    """The restatements on the shapes the GPU file relies on."""
    assert [R.agg_width(n, t, 4096) for n, t in [(1, 8), (1, 9), (1, 32), (1, 33), (4096, 4096 * 100), (2048, 2048 * 100), (2047, 2047 * 33)]] \
        == [4, 8, 8, 32, 4, 8, 32]
    assert [R.norm_per(n) for n in (1, 32767, 32768, 49152, 262143, 262144, 10 ** 7)] == [1, 1, 2, 3, 15, 16, 16]
    off = [0] + [64 * (j + 1) for j in range(64)] + [4096 + 17]
    assert R.h2c_cta_paths(off, True) == [True, True] and R.h2c_cta_paths(off, False) == [False, False]
    assert R.h2c_staged([1] + [4096] * 64, 0, True)                  # counted from the 16-byte word of the first message
    assert not R.h2c_staged([0] * 64 + [4097], 0, True) and not R.h2c_staged([15] + [4097 + 15] * 64, 0, True)


DST_LENGTHS = [0, 1, 21, 22, 54, 55, 56, 85, 86, 119, 120, 255]


def test_host_replay_hash_to_field_lengths(hs):
    """b_0 spans ceil((77 + L + dst_len) / 64) blocks and b_i fits one block only for dst_len <= 21: every message length
    0-129 against each DST length where those boundaries move."""
    for dl in DST_LENGTHS:
        dst = bytes((11 * i + dl) % 256 for i in range(dl))
        for L in range(130):
            msg = bytes((7 * i + L) % 256 for i in range(L))
            out = ctypes.create_string_buffer(192)
            hs.hs_hash_to_field(msg, L, dst, dl, out)
            u = O.hash_to_field_fp2(msg, 2, dst)
            got = ((int.from_bytes(out.raw[0:48], "big"), int.from_bytes(out.raw[48:96], "big")),
                   (int.from_bytes(out.raw[96:144], "big"), int.from_bytes(out.raw[144:192], "big")))
            assert got == (u[0], u[1]), (L, dl)
