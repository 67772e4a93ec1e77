"""hash_to_G2 and the aggregation kernels on every input path their launch code can choose, against the C and Python oracles.

The launch code picks between internal paths from the shape of the input; each rule is restated below and every test builds
its shapes from these restatements and asserts that they land on the path they are meant for:
  - k_hash_to_g2 (kernels.cuh): a CTA hashes B3_TPB / 2 messages and copies their byte range into a shared stage when the range,
    counted from its first 16-byte word, fits B3_H2C_STAGE_BYTES and the blob is 16-byte aligned; otherwise every lane reads
    global memory directly.  sha256_update (h2c.cuh) loads whole words when the input and the block fill are 4-byte aligned.
  - launch_agg (capi.cu): G lanes per set, G in {4, 8, 32}, from (n_sets, total / n_sets, g4_min).
  - norm_per (kernels.cuh): points per inversion of the Jacobian -> affine normalisation.
tests/test_input_paths_cpu.py checks that the constants used here are still the sources'."""
import random

import numpy as np
import pytest

from oracle import bls_oracle as O

pytestmark = pytest.mark.gpu

# ---------------------------------------------------------------- the selection rules, restated
B3_TPB = 128
H2C_MSGS_PER_CTA = B3_TPB // 2                 # two threads per message
H2C_STAGE_BYTES = 4096
AGG_G4_MIN_G1 = 4096                           # kAggG4Min: k_g1_aggregate and k_g1_aggregate_idx
AGG_G4_MIN_G2 = 16384                          # k_g2_aggregate
NORM_POINTS_PER_THREAD = 16384
NORM_MAX = 16


def h2c_staged(off, m0, base_aligned):
    """Whether the CTA whose first message is m0 hashes from the shared stage (off: the n + 1 message offsets)."""
    n = len(off) - 1
    m1 = min(m0 + H2C_MSGS_PER_CTA, n)
    return bool(base_aligned) and int(off[m1]) - (int(off[m0]) & ~15) <= H2C_STAGE_BYTES


def h2c_cta_paths(off, base_aligned):
    return [h2c_staged(off, m0, base_aligned) for m0 in range(0, len(off) - 1, H2C_MSGS_PER_CTA)]


def agg_width(n_sets, total, g4_min):
    avg = total // n_sets
    if n_sets >= g4_min or avg <= 8:
        return 4
    if n_sets >= 2048 or avg <= 32:
        return 8
    return 32


def norm_per(n):
    return min(max(n // NORM_POINTS_PER_THREAD, 1), NORM_MAX)


# ---------------------------------------------------------------- fixtures and helpers
@pytest.fixture(scope="module")
def eng():
    import __graft_entry__ as g
    g.build_cuda()
    import milagro_bls_b200 as mb
    return mb.Engine(0)


def g1w(P):
    return O.serialize_uncompressed_g1(P)


def g2w(P):
    return O.serialize_uncompressed_g2(P)


ONE = O.f12_to_bytes(O.F12_ONE)
_H_CACHE = {}


def c_h2c(m, dst=None):
    """H(m) from the C oracle, memoised (the same messages recur between layouts)."""
    from oracle import c_oracle
    key = (bytes(m), dst)
    if key not in _H_CACHE:
        _H_CACHE[key] = c_oracle.hash_to_g2(m, dst)
    return _H_CACHE[key]


def offsets(msgs):
    return [0] + [int(x) for x in np.cumsum([len(m) for m in msgs])]


def to_dev(b):
    import torch
    a = np.frombuffer(bytes(b), dtype=np.uint8).copy() if not isinstance(b, np.ndarray) else np.ascontiguousarray(b).view(np.uint8).reshape(-1).copy()
    return torch.from_numpy(a).to(torch.device("cuda", 0))


def u32_dev(v):
    return to_dev(np.array(v, dtype=np.uint32))


def msg_bytes(rnd, n):
    return bytes(rnd.getrandbits(8) for _ in range(n))


def check_hashes(out, msgs, py_every=0, dst=None):
    """Every output against the C oracle; every py_every-th message (deterministic) also against the Python oracle."""
    assert out.shape == (len(msgs), 192)
    for j, m in enumerate(msgs):
        assert out[j].tobytes() == c_h2c(m, dst), (j, len(m))
        if py_every and j % py_every == 0:
            assert out[j].tobytes() == g2w(O.hash_to_curve_g2(m, *(() if dst is None else (dst,)))), (j, len(m))


# ---------------------------------------------------------------- 1. message layout matrix (host pointers)
LAYOUT_LENGTHS = list(range(131)) + [191, 192, 255, 256]


def _layout_batch(direct, seed=1):
    """Every length of LAYOUT_LENGTHS at a start offset of every residue mod 16, set by a filler message (0-15 bytes) in front.
    staged layout: a CTA is closed with empty messages before its range would outgrow the stage.  direct layout: the first message
    of every CTA is longer than the stage."""
    rnd, rnd_long = random.Random(seed), random.Random(seed + 1)     # the same targets in both layouts
    msgs, targets = [], []
    total = cta_lo = 0                                                # bytes so far, offset of the current CTA

    def put(m):
        nonlocal total, cta_lo
        if len(msgs) % H2C_MSGS_PER_CTA == 0:
            cta_lo = total
        msgs.append(m)
        total += len(m)

    for r in range(16):
        for L in LAYOUT_LENGTHS:
            pos = len(msgs) % H2C_MSGS_PER_CTA
            if pos > H2C_MSGS_PER_CTA - 2 or (not direct and pos and total + 16 + L - (cta_lo & ~15) > H2C_STAGE_BYTES):
                while len(msgs) % H2C_MSGS_PER_CTA:
                    put(b"")
            if direct and len(msgs) % H2C_MSGS_PER_CTA == 0:
                put(msg_bytes(rnd_long, H2C_STAGE_BYTES + 1 + rnd_long.randrange(16)))
            put(bytes([0xf0 ^ r]) * ((r - total) % 16))
            targets.append(len(msgs))
            put(msg_bytes(rnd, L))
    return msgs, targets


@pytest.mark.parametrize("layout", ["staged", "direct"])
def test_h2c_layout_matrix(eng, layout):
    msgs, targets = _layout_batch(layout == "direct")
    off = offsets(msgs)
    paths = h2c_cta_paths(off, True)
    for t in targets:
        assert paths[t // H2C_MSGS_PER_CTA] == (layout == "staged")
    covered = {(len(msgs[t]), off[t] % 16) for t in targets}
    assert covered == {(L, r) for L in LAYOUT_LENGTHS for r in range(16)}
    out = eng.hash_to_g2(msgs)
    check_hashes(out, msgs)
    for j, t in enumerate(targets):                        # a deterministic subset against the Python oracle
        if j % 29 == 0:
            assert out[t].tobytes() == g2w(O.hash_to_curve_g2(msgs[t])), (len(msgs[t]), off[t] % 16)


def _boundary_batch(ranges, seed=2):
    """CTAs whose byte ranges, counted from the 16-byte word of their first message, are exactly `ranges`; a short tail CTA."""
    rnd = random.Random(seed)
    msgs = []
    lo = 0
    for R in ranges:
        total = R - (lo & 15)
        cuts = sorted(rnd.randrange(total + 1) for _ in range(H2C_MSGS_PER_CTA - 1))
        lens = [b - a for a, b in zip([0] + cuts, cuts + [total])]
        msgs += [msg_bytes(rnd, L) for L in lens]
        lo += total
    msgs += [msg_bytes(rnd, 1 + 3 * k) for k in range(9)]
    return msgs


def test_h2c_stage_boundary(eng):
    ranges = [4096, 4097, 4096, 4097, 4096, 4097, 4097, 4096, 4000]
    msgs = _boundary_batch(ranges)
    off = offsets(msgs)
    paths = h2c_cta_paths(off, True)
    assert paths == [R <= H2C_STAGE_BYTES for R in ranges] + [True]
    cases = {(off[m1] - (off[m0] & ~15), off[m0] % 16 != 0) for m0, m1 in
             ((k * H2C_MSGS_PER_CTA, (k + 1) * H2C_MSGS_PER_CTA) for k in range(len(ranges)))}
    assert {(4096, False), (4096, True), (4097, False), (4097, True)} <= cases
    assert any(a != b for a, b in zip(paths, paths[1:]))
    out = eng.hash_to_g2(msgs)
    check_hashes(out, msgs, py_every=37)


def test_h2c_long_messages(eng):
    rnd = random.Random(3)
    longs = [msg_bytes(rnd, n) for n in (4096, 65536, 1 << 20)]
    for m in longs:                                        # alone: 4 kB still fits the stage, the others do not
        assert h2c_cta_paths([0, len(m)], True) == [len(m) <= H2C_STAGE_BYTES]
        out = eng.hash_to_g2([m])
        check_hashes(out, [m], py_every=1)
    batch = [b"abc"] + longs + [b"z" * 5]                  # unaligned starts, direct path
    assert h2c_cta_paths(offsets(batch), True) == [False]
    check_hashes(eng.hash_to_g2(batch), batch)


# ---------------------------------------------------------------- 2. device entry and misalignment
def test_h2c_dev_entry_every_base_offset(eng):
    import torch
    rnd = random.Random(4)
    msgs = [msg_bytes(rnd, (7 * j) % 71) for j in range(100)]
    off = offsets(msgs)
    blob = b"".join(msgs)
    n = len(msgs)
    buf = torch.zeros(len(blob) + 32, dtype=torch.uint8, device="cuda:0")
    assert buf.data_ptr() % 16 == 0
    d_off = u32_dev(off)
    out = torch.zeros(192 * n, dtype=torch.uint8, device="cuda:0")
    src = to_dev(blob)
    for base in range(16):
        buf.zero_()
        buf[base:base + len(blob)] = src
        aligned = (buf.data_ptr() + base) % 16 == 0
        assert h2c_cta_paths(off, aligned) == [base == 0] * 2
        # word loads of the direct path: on for messages starting at a multiple of 4, off for the others
        assert {(base + off[j]) % 4 for j in range(n) if len(msgs[j]) >= 4} == {0, 1, 2, 3}
        out.fill_(0xAA)
        torch.cuda.synchronize()
        eng.hash_to_g2_dev(buf.data_ptr() + base, d_off.data_ptr(), n, out.data_ptr())
        got = out.cpu().numpy().reshape(n, 192)
        check_hashes(got, msgs, py_every=41 if base in (0, 1, 4) else 0)
    # a misaligned output is refused; n = 0 is a no-op
    with pytest.raises(RuntimeError, match="BadArgument"):
        eng.hash_to_g2_dev(src.data_ptr(), d_off.data_ptr(), n, out.data_ptr() + 4)
    out.fill_(0x5C)
    torch.cuda.synchronize()
    eng.hash_to_g2_dev(src.data_ptr(), d_off.data_ptr(), 0, out.data_ptr())
    assert bool((out == 0x5C).all())
    eng.hash_to_g2_dev(src.data_ptr(), d_off.data_ptr(), n, out.data_ptr())       # the context still works
    check_hashes(out.cpu().numpy().reshape(n, 192), msgs)


# ---------------------------------------------------------------- 3. DST lengths
def _dst(L):
    return bytes((31 * i + 7 + L) % 256 for i in range(L))


def test_h2c_every_dst_length(eng):
    rnd = random.Random(5)
    boundary = {0, 1, 21, 22, 54, 55, 56, 85, 86, 119, 120, 255}
    for L in range(256):
        dst = _dst(L)
        k = L % 8
        msgs = [msg_bytes(rnd, 4 * k + s) for s in (1, 2, 3, 4)]             # msg_len % 4 == 1 absorbs the DST in words
        assert sorted(len(m) % 4 for m in msgs) == [0, 1, 2, 3]
        out = eng.hash_to_g2(msgs, dst=dst)
        check_hashes(out, msgs, dst=dst)
        for j, m in enumerate(msgs):
            if L in boundary or j == L % 4:
                assert out[j].tobytes() == g2w(O.hash_to_curve_g2(m, dst)), (L, len(m))


def test_h2c_oversize_dst_refused(eng):
    import milagro_bls_b200 as mb
    for L in (256, 1000):
        with pytest.raises(mb.AmclError) as e:
            eng.hash_to_g2([b"abc", b"d"], dst=_dst(L))
        assert e.value.kind == "HashToFieldError"
        msgs = [b"abc", b"d" * 77]
        check_hashes(eng.hash_to_g2(msgs, dst=_dst(255)), msgs, dst=_dst(255))
        check_hashes(eng.hash_to_g2(msgs), msgs, py_every=1)


# ---------------------------------------------------------------- 4. hashing inside verification
def _signed(eng, msgs, rnd):
    """(sks, pks (n, 96), sigs (n, 192)): sig_i = [sk_i] H(m_i) with H(m_i) from the C oracle."""
    sks = [rnd.randrange(1, O.r) for _ in msgs]
    pks = eng.g1_mul_gen(sks)
    H = b"".join(c_h2c(m) for m in msgs)
    return sks, pks, eng.g2_mul(H, sks)


def _flip_last(msgs):
    m = msgs[-1]
    return msgs[:-1] + [m[:-1] + bytes([m[-1] ^ 1])]


def test_verify_long_message(eng):
    from oracle import c_oracle
    rnd = random.Random(6)
    m = msg_bytes(rnd, 10 * 1024)
    assert h2c_cta_paths([0, len(m)], True) == [False]
    _, pks, sigs = _signed(eng, [m], rnd)
    ok, gt = eng.verify(sigs[0].tobytes(), pks[0].tobytes(), m, want_gt=True)
    assert ok and gt == ONE
    bad = _flip_last([m])[0]
    ok, gt = eng.verify(sigs[0].tobytes(), pks[0].tobytes(), bad, want_gt=True)
    ok_c, gt_c = c_oracle.fast_aggregate_verify(sigs[0].tobytes(), pks[0].tobytes(), bad, reject_inf=False)
    assert not ok and not ok_c and gt == gt_c != ONE


def test_aggregate_verify_direct_path(eng):
    from oracle import c_oracle
    rnd = random.Random(7)
    msgs = [msg_bytes(rnd, rnd.randrange(100, 301)) for _ in range(70)]
    assert h2c_cta_paths(offsets(msgs), True)[0] is False
    _, pks, sigs = _signed(eng, msgs, rnd)
    agg = g2w(O.aggregate_signatures([O.deserialize_g2(s.tobytes()) for s in sigs]))
    ok, gt = eng.aggregate_verify(agg, pks.reshape(-1), msgs, want_gt=True)
    assert ok and gt == ONE
    bad = _flip_last(msgs)
    ok, gt = eng.aggregate_verify(agg, pks.reshape(-1), bad, want_gt=True)
    ok_c, gt_c = c_oracle.aggregate_verify(agg, pks.reshape(-1), bad)
    assert not ok and not ok_c and gt == gt_c != ONE


def test_verify_multiple_direct_path(eng):
    from oracle import c_oracle
    rnd = random.Random(8)
    n = 130
    msgs = [msg_bytes(rnd, 100) for _ in range(n)]
    moff = offsets(msgs)
    assert h2c_cta_paths(moff, True) == [False, False, True]
    _, pks, sigs = _signed(eng, msgs, rnd)
    scalars = np.array([rnd.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    ok, fb, gt = eng.verify_multiple(sigs.reshape(-1), pks.reshape(-1), None, b"".join(msgs), moff, scalars, want_gt=True)
    assert ok and fb == -1 and gt == ONE
    bad = b"".join(_flip_last(msgs))
    ok, fb, gt = eng.verify_multiple(sigs.reshape(-1), pks.reshape(-1), None, bad, moff, scalars, want_gt=True)
    ok_c, gt_c = c_oracle.verify_multiple(sigs.reshape(-1), pks.reshape(-1), None, bad, moff, scalars)
    assert not ok and not ok_c and fb == -1 and gt == gt_c != ONE


def test_verify_batch_direct_path(eng):
    from oracle import c_oracle
    from milagro_bls_b200 import _lib
    rnd = random.Random(9)
    msgs = [msg_bytes(rnd, rnd.randrange(100, 301)) for _ in range(70)]
    assert h2c_cta_paths(offsets(msgs), True)[0] is False
    _, pks, sigs = _signed(eng, msgs, rnd)
    acc, st, gt = eng.verify_batch(_lib.ITEM_VERIFY, sigs.reshape(-1), pks.reshape(-1), None, msgs, want_gt=True)
    assert acc.all() and not st.any() and all(g.tobytes() == ONE for g in gt)
    bad = _flip_last(msgs)
    acc, st, gt = eng.verify_batch(_lib.ITEM_VERIFY, sigs.reshape(-1), pks.reshape(-1), None, bad, want_gt=True)
    assert list(np.nonzero(~acc)[0]) == [69] and not st.any()
    assert all(gt[i].tobytes() == ONE for i in range(69))
    ok_c, gt_c = c_oracle.fast_aggregate_verify(sigs[69].tobytes(), pks[69].tobytes(), bad[69], reject_inf=False)
    assert not ok_c and gt[69].tobytes() == gt_c


def test_verify_multiple_grouped_long_messages(eng):
    from oracle import c_oracle
    rnd = random.Random(10)
    distinct = [msg_bytes(rnd, 1500 + 7 * k) for k in range(4)]
    dmoff = offsets(distinct)
    assert h2c_cta_paths(dmoff, True) == [False]
    n = 12
    idx = [j % 4 for j in range(n)]
    sks = [rnd.randrange(1, O.r) for _ in range(2 * n)]
    pks = eng.g1_mul_gen(sks)
    H = b"".join(c_h2c(distinct[k]) for k in idx)
    sigs = eng.g2_mul(H, [(sks[2 * j] + sks[2 * j + 1]) % O.r for j in range(n)])
    pk_off = list(range(0, 2 * n + 1, 2))
    scalars = np.array([rnd.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    ok, fb, gt = eng.verify_multiple_grouped(None, sigs.reshape(-1), pks.reshape(-1), pk_off, b"".join(distinct), dmoff, idx, scalars,
                                             want_gt=True)
    assert ok and fb == -1 and gt == ONE
    bad = _flip_last(distinct)
    ok, fb, gt = eng.verify_multiple_grouped(None, sigs.reshape(-1), pks.reshape(-1), pk_off, b"".join(bad), dmoff, idx, scalars,
                                             want_gt=True)
    expanded = [bad[k] for k in idx]
    ok_c, gt_c = c_oracle.verify_multiple(sigs.reshape(-1), pks.reshape(-1), pk_off, b"".join(expanded), offsets(expanded), scalars)
    assert not ok and not ok_c and fb == -1 and gt == gt_c != ONE


# ---------------------------------------------------------------- 5. aggregation widths x edge placement
POOL = 24


@pytest.fixture(scope="module")
def pools():
    """Random points of G1 and G2 (from the C oracle) and their wire forms."""
    from oracle import c_oracle
    rnd = random.Random(12)
    g1 = [O.deserialize_g1(c_oracle.g1_mul(g1w(O.G1_GEN), rnd.randrange(1, O.r))) for _ in range(POOL)]
    g2 = [O.deserialize_g2(c_oracle.g2_mul(g2w(O.G2_GEN), rnd.randrange(1, O.r))) for _ in range(POOL)]
    return g1, g2


def _edge_sets(G, rnd):
    """Edge sets for G lanes per set, as lists of tokens: ("P", k) pool point k, ("N", k) its negative, ("I",) infinity,
    ("B", kind) a bad record.  Returns (name, tokens) pairs."""
    def fill(n):
        return [("P", rnd.randrange(POOL)) for _ in range(n)]

    def at(n, where):
        s = fill(n)
        for i, t in where.items():
            s[i] = t
        return s

    a, b = rnd.randrange(POOL), rnd.randrange(POOL)
    while b == a:
        b = rnd.randrange(POOL)
    P, N = ("P", a), ("N", a)
    sets = [
        ("empty_first", []),
        ("dbl_mixed_lane0", at(2 * G + 1, {0: P, G: P})),
        ("dbl_mixed_lane_last", at(2 * G + 1, {G - 1: P, 2 * G - 1: P})),
        ("dbl_tree", [P, P]),
        ("dbl_tree_in_set", at(G, {0: P, G // 2: P})),
        ("lanes_equal", [P] * G),
        ("lanes_equal_twice", [P] * (2 * G)),
        ("cancel_mixed", at(G + 1, {0: P, G: N})),
        ("cancel_mixed_all", [("P", (a + i) % POOL) for i in range(G)] + [("N", (a + i) % POOL) for i in range(G)]),
        ("cancel_tree", [P, N]),
        ("cancel_tree_2", [P, ("P", b), N, ("N", b)]),
        ("cancel_runs", [P] * 5 + [N] * 5),
        ("empty_middle", []),
        ("inf_one", [("I",)]),
        ("inf_all", [("I",)] * (G + 1)),
        ("inf_lane0_strides", at(2 * G + 1, {0: ("I",), G: ("I",), 2 * G: ("I",), G - 1: ("I",)})),
        ("len_G-1", fill(G - 1)),
        ("len_G", fill(G)),
        ("len_G+1", fill(G + 1)),
        ("len_2G+1", fill(2 * G + 1)),
    ]
    for kind in ("off_curve", "cflag", "range"):
        sets.append((f"before_bad_{kind}", fill(G + 1)))
        sets.append((f"bad_{kind}", at(2 * G + 1, {2 * G - 1: ("B", kind)})))      # second stride of lane G - 1
        sets.append((f"after_bad_{kind}", fill(2 * G + 1)))
    sets.append(("empty_last", []))
    return sets


class _Kernel:
    """One aggregation kernel: renders token sets to its input form and computes the expected results."""

    def __init__(self, name, eng, pools):
        self.name, self.eng = name, eng
        g1, g2 = pools
        self.g2 = name == "g2"
        self.pts = g2 if self.g2 else g1
        self.neg = O.g2_neg if self.g2 else O.g1_neg
        self.w = g2w if self.g2 else g1w
        self.g4_min = AGG_G4_MIN_G2 if self.g2 else AGG_G4_MIN_G1
        self.bad_kinds = ("range",) if name == "g1_idx" else ("off_curve", "cflag")
        self.table = None
        if name == "g1_idx":
            import milagro_bls_b200 as mb
            self.table = mb.KeyTable(eng)
            recs = [g1w(P) for P in g1] + [g1w(O.g1_neg(P)) for P in g1] + [g1w(None)]
            first, st = self.table.append(b"".join(recs), compressed=False, validate=False)
            assert first == 0 and not st.any()

    def edge_sets(self, G, rnd):
        """_edge_sets with the bad records this kernel can receive"""
        return [(n, s) for n, s in _edge_sets(G, rnd) if not any(n.endswith(k) for k in ("off_curve", "cflag", "range") if k not in self.bad_kinds)]

    def point(self, t):
        return {"P": lambda: self.pts[t[1]], "N": lambda: self.neg(self.pts[t[1]]), "I": lambda: None}[t[0]]()

    def render(self, t):
        if self.name == "g1_idx":
            if t[0] == "B":
                return 3 * POOL + 1000                      # out of range of the table
            return 2 * POOL if t[0] == "I" else t[1] + (POOL if t[0] == "N" else 0)
        if t[0] == "B":
            rec = bytearray(self.w(self.pts[0]))
            if t[1] == "off_curve":
                rec[-1] ^= 1
            else:
                rec[0] |= 0x80                              # compressed flag on an uncompressed record
            return bytes(rec)
        return self.w(self.point(t))

    def run(self, sets):
        recs = [self.render(t) for s in sets for t in s]
        off = offsets(sets)
        if self.name == "g1_idx":
            out, st = self.eng.g1_aggregate_indexed(self.table, np.array(recs, dtype=np.uint32), off)
        elif self.g2:
            out, st = self.eng.g2_aggregate(b"".join(recs), off)
        else:
            out, st = self.eng.g1_aggregate(b"".join(recs), off)
        rec_bytes = 192 if self.g2 else 96
        return out.reshape(len(sets), rec_bytes), st

    def expected(self, s):
        """(status, wire bytes or None when the bytes are not part of the contract)"""
        if any(t[0] == "B" for t in s):
            return -5, None
        if not s:
            return (0, g2w(None)) if self.g2 else (-1, None)
        if self.g2:
            return 0, g2w(O.aggregate_signatures([self.point(t) for t in s]))
        from oracle import c_oracle
        rc, w = c_oracle.g1_aggregate(b"".join(g1w(self.point(t)) for t in s))
        assert rc == 0
        return 0, w


@pytest.mark.parametrize("G", [4, 8, 32])
@pytest.mark.parametrize("kernel", ["g1", "g1_idx", "g2"])
def test_aggregate_edges_at_every_width(eng, pools, kernel, G):
    K = _Kernel(kernel, eng, pools)
    rnd = random.Random(100 + G)
    named = K.edge_sets(G, rnd)
    filler = {4: 1, 8: 30, 32: 120}[G]
    for _ in range(200):                                      # fillers move the average set size to the width under test
        total = sum(len(s) for _, s in named)
        if agg_width(len(named), total, K.g4_min) == G:
            break
        named.append((f"filler{len(named)}", [("P", rnd.randrange(POOL)) for _ in range(filler)]))
    assert agg_width(len(named), sum(len(s) for _, s in named), K.g4_min) == G
    sets = [s for _, s in named]
    out, st = K.run(sets)
    for j, (name, s) in enumerate(named):
        code, w = K.expected(s)
        assert st[j] == code, (name, int(st[j]))
        if w is not None:
            assert out[j].tobytes() == w, name


def test_aggregate_signature_api_sizes(eng, pools):
    import milagro_bls_b200 as mb
    g2 = pools[1]
    rnd = random.Random(13)
    widths = set()
    for n in (1, 8, 9, 32, 33, 200):
        pts = [g2[rnd.randrange(POOL)] for _ in range(n)]
        widths.add(agg_width(1, n, AGG_G4_MIN_G2))
        agg = mb.AggregateSignature.aggregate([mb.Signature(g2w(P)) for P in pts], engine=eng)
        assert agg.point == g2w(O.aggregate_signatures(pts)), n
    assert widths == {4, 8, 32}


def test_g1_aggregate_dev_entry(eng, pools):
    import torch
    K = _Kernel("g1", eng, pools)
    sets = [s for _, s in K.edge_sets(8, random.Random(14))]
    recs = b"".join(K.render(t) for s in sets for t in s)
    off = offsets(sets)
    n = len(sets)
    ref_out, ref_st = eng.g1_aggregate(recs, off)
    d_pks, d_off = to_dev(recs), u32_dev(off)
    out = torch.zeros(96 * n, dtype=torch.uint8, device="cuda:0")
    st = torch.zeros(n, dtype=torch.int32, device="cuda:0")
    torch.cuda.synchronize()
    eng.g1_aggregate_dev(d_pks.data_ptr(), d_off.data_ptr(), n, out.data_ptr(), st.data_ptr())
    assert out.cpu().numpy().tobytes() == ref_out.tobytes()
    assert list(st.cpu().numpy()) == list(ref_st)
    for j, s in enumerate(sets):
        code, w = K.expected(s)
        assert ref_st[j] == code and (w is None or ref_out[96 * j:96 * j + 96].tobytes() == w), j
    big = torch.zeros(len(recs) + 16, dtype=torch.uint8, device="cuda:0")
    for bad_pks, bad_out in ((big.data_ptr() + 8, out.data_ptr()), (d_pks.data_ptr(), out.data_ptr() + 8)):
        with pytest.raises(RuntimeError, match="BadArgument"):
            eng.g1_aggregate_dev(bad_pks, d_off.data_ptr(), n, bad_out, st.data_ptr())


def test_keytable_get_out_of_range(eng, pools):
    g1 = pools[0]
    K = _Kernel("g1_idx", eng, pools)
    n_table = len(K.table)
    idx = [0, n_table - 1, n_table, 5, 0xFFFFFFFF, n_table + 7, 2 * POOL]
    out, st = K.table.get(idx)
    want = {0: g1w(g1[0]), n_table - 1: g1w(None), 5: g1w(g1[5]), 2 * POOL: g1w(None)}
    for j, k in enumerate(idx):
        if k in want:
            assert st[j] == 0 and out[j].tobytes() == want[k], k
        else:
            assert st[j] == -5 and out[j].tobytes() == bytes(96), k


# ---------------------------------------------------------------- 6. normalisation chunks
@pytest.mark.parametrize("n_sets", [32767, 32768, 262144 + 7])
@pytest.mark.parametrize("group", ["g1", "g2"])
def test_normalisation_chunks(eng, pools, group, n_sets):
    """Every set of a large call is one of four kinds over a small pool -- one point, two points, P + (-P), an infinity record
    -- so its expected value is known by construction.  Infinities sit at the first and the last slot of chunks of norm_per
    points, one chunk is all infinities, and at 262151 sets the last chunk is short."""
    is_g2 = group == "g2"
    pts = pools[1] if is_g2 else pools[0]
    W = 192 if is_g2 else 96
    wire = g2w if is_g2 else g1w
    neg = O.g2_neg if is_g2 else O.g1_neg
    add = O.g2_add if is_g2 else O.g1_add
    per = norm_per(n_sets)
    assert per == {32767: 1, 32768: 2, 262151: 16}[n_sets]
    assert n_sets % per == (7 if n_sets == 262151 else 0)                 # a short last chunk at per = 16
    # record table: pool, negated pool, infinity; expected table: pool, pair sums, infinity
    rec_tab = np.frombuffer(b"".join([wire(P) for P in pts] + [wire(neg(P)) for P in pts] + [wire(None)]), dtype=np.uint8).reshape(-1, W)
    exp_tab = np.frombuffer(b"".join([wire(P) for P in pts] + [wire(add(P, pts[(k + 1) % POOL])) for k, P in enumerate(pts)]
                                     + [wire(None)]), dtype=np.uint8).reshape(-1, W)
    INF = 2 * POOL
    rng = np.random.default_rng(n_sets)
    kind = rng.integers(0, 4, n_sets)                     # 0 one point, 1 two points, 2 P + (-P), 3 infinity record
    k = rng.integers(0, POOL, n_sets)
    n_chunks = (n_sets + per - 1) // per
    first = np.arange(0, n_chunks, 5) * per               # first slot of every 5th chunk, last slot of every 7th
    last = np.minimum(np.arange(3, n_chunks, 7) * per + per - 1, n_sets - 1)
    kind[first] = np.where(np.arange(len(first)) % 2, 2, 3)
    kind[last] = np.where(np.arange(len(last)) % 2, 3, 2)
    all_inf = 6 * per + np.arange(per)                    # chunk 6: every slot infinite
    kind[all_inf] = 3
    kind[n_sets - 1] = 0                                   # the short last chunk ends on a finite point
    counts = np.array([1, 2, 2, 1])[kind]
    off = np.concatenate([[0], np.cumsum(counts)]).astype(np.uint32)
    rec = np.empty(int(off[-1]), dtype=np.int64)
    rec[off[:-1]] = np.where(kind == 3, INF, k)
    two = counts == 2
    rec[off[:-1][two] + 1] = np.where(kind[two] == 1, (k[two] + 1) % POOL, POOL + k[two])
    exp_idx = np.where(kind == 0, k, np.where(kind == 1, POOL + k, INF))
    assert agg_width(n_sets, int(off[-1]), AGG_G4_MIN_G2 if is_g2 else AGG_G4_MIN_G1) == 4
    blob = rec_tab[rec].reshape(-1)
    out, st = (eng.g2_aggregate if is_g2 else eng.g1_aggregate)(blob, off)
    assert not st.any()
    got = out.reshape(n_sets, W)
    bad = np.nonzero((got != exp_tab[exp_idx]).any(axis=1))[0]
    assert len(bad) == 0, (len(bad), bad[:10], kind[bad[:10]])


# ---------------------------------------------------------------- 7. b3_verify_batch_dev
def _batch_items():
    """A mixed bag of items: (sig point, [key points], msg).  Valid, wrong message, wrong key, non-subgroup signature,
    signature at infinity, key at infinity, keys summing to infinity, empty key list, ragged messages."""
    sks = [4242 + 17 * i for i in range(5)]
    pks_o = [O.sk_to_pk(s) for s in sks]
    items = []
    for j, m in enumerate([b"", b"a", b"cats", bytes(range(32)), bytes(200)]):
        ks = list(range(1 + j % 4))
        sig = O.aggregate_signatures([O.sign(sks[k], m) for k in ks])
        items.append((sig, [pks_o[k] for k in ks], m))
    sig, ks, m = items[2]
    items.append((sig, ks, b"dogs"))                                         # wrong message
    items.append((sig, ks[:-1] + [pks_o[4]], m))                             # wrong key
    items.append((O.map_to_curve_g2((5, 7)), ks, m))                         # on curve, not in G2
    items.append((None, ks, m))                                              # signature at infinity
    items.append((sig, [None], m))                                           # key at infinity
    items.append((None, [O.sk_to_pk(1), O.sk_to_pk(O.r - 1)], m))            # keys sum to infinity, sig = infinity
    items.append((sig, [], m))                                               # no keys
    return items


def test_verify_batch_dev_matches_host(eng):
    import torch
    from milagro_bls_b200 import _lib
    items = _batch_items()
    n = len(items)
    sigs = b"".join(g2w(s) for s, _, _ in items)
    pks = b"".join(g1w(P) for _, ks, _ in items for P in ks)
    pk_off = offsets([ks for _, ks, _ in items])
    msgs = [m for _, _, m in items]
    acc_h, st_h, gt_h = eng.verify_batch(_lib.ITEM_FAST_AGGREGATE, sigs, pks, pk_off, msgs, want_gt=True)
    assert acc_h.sum() == 5
    blob = b"".join(msgs)
    moff = offsets(msgs)
    d_sigs, d_pks, d_pk_off, d_moff = to_dev(sigs), to_dev(pks), u32_dev(pk_off), u32_dev(moff)
    buf = torch.zeros(len(blob) + 16, dtype=torch.uint8, device="cuda:0")
    for base in (0, 3):                                   # staged, and a misaligned blob (direct path)
        if blob:
            buf[base:base + len(blob)] = to_dev(blob)
        assert h2c_cta_paths(moff, (buf.data_ptr() + base) % 16 == 0) == [base == 0]
        acc = torch.full((n,), 7, dtype=torch.int32, device="cuda:0")
        st = torch.full((n,), 7, dtype=torch.int32, device="cuda:0")
        gt = torch.full((n * 576,), 0xEE, dtype=torch.uint8, device="cuda:0")
        torch.cuda.synchronize()
        eng.verify_batch_dev(_lib.ITEM_FAST_AGGREGATE, d_sigs.data_ptr(), d_pks.data_ptr(), d_pk_off.data_ptr(), buf.data_ptr() + base,
                             d_moff.data_ptr(), n, acc.data_ptr(), st.data_ptr(), gt.data_ptr())
        assert [bool(a) for a in acc.cpu().numpy()] == list(acc_h), base
        assert list(st.cpu().numpy()) == list(st_h), base
        assert gt.cpu().numpy().tobytes() == gt_h.tobytes(), base
