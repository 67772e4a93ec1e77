"""b3_verify_multiple_grouped: verify_multiple over sets that name their message by index, each distinct message hashed and
paired once.  Its accept bit, first_bad and all 576 GT bytes must equal those of b3_verify_multiple / _indexed on the same sets
with every set's message written out (the expanded call), for

  * message shapes: every set its own message (identity and permuted msg_idx), one message for all sets, mixed group sizes
    (one dominant group and singletons), unreferenced messages, groups whose scaled keys sum to infinity;
  * sizes either side of the signature-MSM switch (512 sets), 512 x 1 key on one message, 8192 x 1 key over 64 messages and
    8192 x 128 table keys over 64 messages;
  * byte keys and table keys (an invalid table entry gives _indexed's error), host and device pointers, the precheck flow,
    latency modes and serial / overlapped stages;
  * rejections in a large group (tampered signature, wrong key, non-subgroup signature);
  * argument errors (n_msgs == 0, msg_idx out of range with host and device pointers, a zero scalar), after which the context
    still gives correct results;
  * b3_verify_multiple_locate after a grouped call, and the Python extension (result and RNG state of the ungrouped function).
"""
import random

import numpy as np
import pytest

from oracle import bls_oracle as O
from oracle import c_oracle

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def eng():
    import __graft_entry__ as g
    g.build_cuda()
    import milagro_bls_b200 as mb
    e = mb.Engine(0)
    mb.set_default_engine(e)
    return e


def g1w(P):
    return O.serialize_uncompressed_g1(P)


def g2w(P):
    return O.serialize_uncompressed_g2(P)


def u8(b):
    return np.frombuffer(bytes(b), dtype=np.uint8)


def _offs(chunks):
    return np.array([0] + list(np.cumsum([len(c) for c in chunks])), dtype=np.uint32)


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).to(torch.device("cuda", 0))


def _synth(eng, n, nk, msg_idx, n_msgs, seed):
    """n valid sets of nk keys each; set j signs message msg_idx[j] of n_msgs 32-byte messages."""
    rnd = random.Random(seed)
    pool_n = max(4 * nk, 64)
    sks = [rnd.randrange(1, O.r) for _ in range(pool_n)]
    pool = eng.g1_mul_gen(sks)
    rs = np.random.RandomState(seed & 0xffff)
    idx = np.stack([rs.choice(pool_n, size=nk, replace=False) for _ in range(n)]).astype(np.uint32)
    msgs = rs.randint(0, 256, size=(n_msgs, 32), dtype=np.uint8)
    msgs[:, :4] = np.arange(n_msgs, dtype=">u4").view(np.uint8).reshape(n_msgs, 4)
    agg_sk = [sum(sks[i] for i in row) % O.r for row in idx]
    mi = np.asarray(msg_idx, dtype=np.uint32)
    H = eng.hash_to_g2([m.tobytes() for m in msgs])
    sigs = eng.g2_mul(np.ascontiguousarray(H[mi]).reshape(-1), agg_sk)
    scalars = np.array([rnd.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    return {"n": n, "nk": nk, "pool": pool, "idx": idx, "pks": np.ascontiguousarray(pool[idx.reshape(-1)]).reshape(-1),
            "pk_off": np.arange(0, n * nk + 1, nk, dtype=np.uint32), "msgs": [m.tobytes() for m in msgs], "mi": mi,
            "sigs": np.ascontiguousarray(sigs).reshape(-1), "scalars": scalars}


def _grouped(eng, b, sigs=None, table=None, keys=None, mi=None, scalars=None, msgs=None):
    msgs = b["msgs"] if msgs is None else msgs
    return eng.verify_multiple_grouped(table, b["sigs"] if sigs is None else sigs, b["pks"] if keys is None else keys, b["pk_off"],
                                       b"".join(msgs), _offs(msgs), b["mi"] if mi is None else mi,
                                       b["scalars"] if scalars is None else scalars, want_gt=True)


def _expanded(eng, b, sigs=None, table=None, keys=None, mi=None, scalars=None, msgs=None):
    msgs = b["msgs"] if msgs is None else msgs
    ex = [msgs[k] for k in (b["mi"] if mi is None else mi)]
    args = (b["pk_off"], b"".join(ex), _offs(ex), b["scalars"] if scalars is None else scalars)
    sigs = b["sigs"] if sigs is None else sigs
    if table is None:
        return eng.verify_multiple(sigs, b["pks"] if keys is None else keys, *args, want_gt=True)
    return eng.verify_multiple_indexed(table, sigs, keys, *args, want_gt=True)


def _same(eng, b, **kw):
    g = _grouped(eng, b, **kw)
    x = _expanded(eng, b, **kw)
    assert g == x
    return g


def _shapes(n, rs):
    """(name, msg_idx, n_msgs) for the message shapes of a batch of n sets."""
    dom = np.zeros(n, dtype=np.uint32)                           # one dominant group, then singletons
    k = max(n // 8, 1)
    dom[n - k:] = np.arange(1, k + 1)
    unref = (np.arange(n) % 3 * 2 + 1).astype(np.uint32)       # messages 1, 3, 5 named; 0, 2, 4, 6 not
    return [("identity", np.arange(n, dtype=np.uint32), n),
            ("permuted", rs.permutation(n).astype(np.uint32), n),
            ("one message", np.zeros(n, dtype=np.uint32), 1),
            ("dominant and singletons", dom, k + 1),
            ("random groups", rs.randint(0, max(n // 4, 1), size=n).astype(np.uint32), max(n // 4, 1)),
            ("unreferenced", unref, 7)]


@pytest.mark.parametrize("n", [5, 511, 512, 513])
def test_message_shapes(eng, n):
    rs = np.random.RandomState(n)
    for name, mi, n_msgs in _shapes(n, rs):
        b = _synth(eng, n, 2, mi, n_msgs, 0x6A0 + n)
        ok, fb, gt = _same(eng, b)
        assert ok and fb == -1, name
        if n == 5:
            ex = [b["msgs"][k] for k in mi]
            assert c_oracle.verify_multiple(b["sigs"], b["pks"], b["pk_off"], b"".join(ex), _offs(ex), b["scalars"])[0], name
        # one tampered signature in the largest group is rejected exactly as the expanded call rejects it
        j = int(np.argmax(np.bincount(mi, minlength=n_msgs)[mi]))
        sigs = b["sigs"].copy()
        sigs[192 * j:192 * (j + 1)] = b["sigs"][192 * ((j + 1) % n):192 * ((j + 1) % n + 1)]
        ok, fb, _ = _same(eng, b, sigs=sigs)
        assert not ok and fb == -1, name


def test_infinite_groups(eng):
    """Groups whose scaled keys sum to infinity: keys P and -P with equal scalars in one group, an empty key range, keys that
    cancel inside a set -- each contributes 1 -- next to a group of valid sets; and a message that no set names."""
    rnd = random.Random(0x1AF)
    sk = [rnd.randrange(1, O.r) for _ in range(4)]
    pk = [O.sk_to_pk(s) for s in sk]
    m = [b"grouped infinity %d" % k for k in range(4)]
    sets = [(O.sign(sk[0], m[0]), [pk[0]], 0), (O.g2_neg(O.sign(sk[0], m[0])), [O.g1_neg(pk[0])], 0),    # P, -P: same scalar
            (None, [], 1), (None, [pk[1], O.g1_neg(pk[1])], 1),                                          # empty range, cancelling keys
            (O.sign(sk[2], m[2]), [pk[2]], 2), (O.sign(sk[3], m[2]), [pk[3]], 2), (O.sign(sk[2], m[2]), [pk[2]], 2)]   # equal points
    n = len(sets)
    b = {"sigs": u8(b"".join(g2w(s) for s, _, _ in sets)), "pks": u8(b"".join(g1w(P) for _, ks, _ in sets for P in ks)),
         "pk_off": _offs([[0] * len(ks) for _, ks, _ in sets]), "msgs": m, "mi": np.array([k for _, _, k in sets], dtype=np.uint32)}
    sc = np.array([rnd.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    sc[1] = sc[0]
    sc[6] = sc[4]
    b["scalars"] = sc
    ok, fb, gt = _same(eng, b)
    assert ok and fb == -1
    ex = [m[k] for k in b["mi"]]
    assert c_oracle.verify_multiple(b["sigs"], b["pks"], b["pk_off"], b"".join(ex), _offs(ex), sc)[0]
    # only the cancelling group: the whole product is 1
    sub = {"sigs": b["sigs"][:384], "pks": b["pks"][:192], "pk_off": b["pk_off"][:3], "msgs": m, "mi": b["mi"][:2], "scalars": sc[:2]}
    ok, fb, gt = _same(eng, sub)
    assert ok and fb == -1


@pytest.fixture(scope="module")
def big(eng):
    """8192 sets x 1 key over 64 messages."""
    rs = np.random.RandomState(64)
    return _synth(eng, 8192, 1, rs.randint(0, 64, size=8192), 64, 0xB16)


def test_large_group_shapes(eng, big):
    ok, fb, gt = _same(eng, big)
    assert ok and fb == -1
    b512 = _synth(eng, 512, 1, np.zeros(512, dtype=np.uint32), 1, 0x512)
    ok, fb, gt = _same(eng, b512)
    assert ok and fb == -1
    # one group of every set (8192 sets on one message: a log-depth tree)
    one = dict(big)
    one["mi"] = np.zeros(8192, dtype=np.uint32)
    one["msgs"] = [big["msgs"][0]]
    ok, fb, gt = _same(eng, one)
    assert not ok and fb == -1


def test_rejections_in_a_large_group(eng, big):
    ns = np.frombuffer(g2w(O.map_to_curve_g2((5, 7))), dtype=np.uint8)
    g = int(np.bincount(big["mi"]).argmax())
    members = np.flatnonzero(big["mi"] == g)
    j0, j1, j2 = int(members[3]), int(members[len(members) // 2]), int(members[-2])
    sigs = big["sigs"].copy()                                    # tampered: another member's signature
    sigs[192 * j0:192 * (j0 + 1)] = big["sigs"][192 * j1:192 * (j1 + 1)]
    ok, fb, _ = _same(eng, big, sigs=sigs)
    assert not ok and fb == -1
    pks = big["pks"].copy()                                      # wrong key
    pks[96 * j2:96 * (j2 + 1)] = big["pool"][(int(big["idx"][j2, 0]) + 1) % len(big["pool"])]
    ok, fb, _ = _same(eng, big, keys=pks)
    assert not ok and fb == -1
    sigs = big["sigs"].copy()                                    # non-subgroup signature
    sigs[192 * j1:192 * (j1 + 1)] = ns
    ok, fb, _ = _same(eng, big, sigs=sigs)
    assert not ok and fb == j1


@pytest.fixture(scope="module")
def c4g(eng):
    """8192 sets x 128 table keys over 64 messages, from a pool of 4096 validators."""
    rs = np.random.RandomState(0xC46)
    return _synth(eng, 8192, 128, rs.randint(0, 64, size=8192), 64, 0xC4C4)


def test_table_keys_8192x128(eng, c4g):
    import milagro_bls_b200 as mb
    b = c4g
    tbl = mb.KeyTable(eng)
    _, st = tbl.append(b["pool"].reshape(-1), compressed=False, validate=True)
    assert not st.any()
    kidx = b["idx"].reshape(-1)
    ok, fb, gt = _same(eng, b, table=tbl, keys=kidx)
    assert ok and fb == -1
    assert _grouped(eng, b) == (ok, fb, gt)                     # byte keys: the same bytes
    # an invalid table entry: the error of _indexed
    bad = np.zeros(96, dtype=np.uint8)
    bad[0] = 0x01                                               # not on the curve: appended, marked invalid
    first, st = tbl.append(bad, compressed=False, validate=True)
    assert st[0] != 0
    k2 = kidx.copy()
    k2[128 * 4000 + 7] = first
    with pytest.raises(Exception) as eg:
        _grouped(eng, b, table=tbl, keys=k2)
    with pytest.raises(Exception) as ex:
        _expanded(eng, b, table=tbl, keys=k2)
    assert type(eg.value) is type(ex.value) and str(eg.value) == str(ex.value)
    assert _grouped(eng, b, table=tbl, keys=kidx) == (ok, fb, gt)


def test_device_pointers_precheck_modes(eng, big):
    b = big
    want = _expanded(eng, b)
    d = [_dev(a) for a in (b["sigs"], b["pks"], u8(b"".join(b["msgs"])), _offs(b["msgs"]), b["mi"], b["scalars"])]
    got = eng.verify_multiple_grouped_dev(None, d[0].data_ptr(), d[1].data_ptr(), 0, d[2].data_ptr(), d[3].data_ptr(), 64, d[4].data_ptr(),
                                          d[5].data_ptr(), b["n"], want_gt=True)
    assert got == want
    # the precheck flow: sigs192 None reuses the checked signatures
    assert eng.sig_precheck(b["sigs"]) == -1
    assert eng.verify_multiple_grouped(None, None, b["pks"], None, b"".join(b["msgs"]), _offs(b["msgs"]), b["mi"], b["scalars"],
                                       want_gt=True) == want
    # latency modes, serial / overlapped: identical bytes
    try:
        for mode in (0, 1, 2):
            for serial in (False, True):
                eng.set_latency_mode(mode)
                eng.set_serial(serial)
                assert _grouped(eng, b) == want, (mode, serial)
    finally:
        eng.set_latency_mode(0)
        eng.set_serial(False)


def test_argument_errors(eng, big):
    b = big
    want = _grouped(eng, b)
    blob, off = b"".join(b["msgs"]), _offs(b["msgs"])
    with pytest.raises(RuntimeError, match="BadArgument"):       # n_msgs == 0
        eng.verify_multiple_grouped(None, b["sigs"], b["pks"], b["pk_off"], b"", [0], b["mi"], b["scalars"])
    mi = b["mi"].copy()
    mi[4321] = 64
    with pytest.raises(RuntimeError, match="BadArgument"):       # out of range, host pointers
        eng.verify_multiple_grouped(None, b["sigs"], b["pks"], b["pk_off"], blob, off, mi, b["scalars"])
    assert _grouped(eng, b) == want
    d = [_dev(a) for a in (b["sigs"], b["pks"], u8(blob), off, mi, b["scalars"])]
    with pytest.raises(RuntimeError, match="BadArgument"):       # out of range, device pointers: the device flag
        eng.verify_multiple_grouped_dev(None, d[0].data_ptr(), d[1].data_ptr(), 0, d[2].data_ptr(), d[3].data_ptr(), 64, d[4].data_ptr(),
                                        d[5].data_ptr(), b["n"])
    with pytest.raises(RuntimeError, match="BadArgument"):
        eng.verify_multiple_locate(b["n"])
    assert _grouped(eng, b) == want
    sc = b["scalars"].copy()
    sc[77] = 0
    with pytest.raises(RuntimeError, match="BadArgument"):       # zero scalar
        _grouped(eng, b, scalars=sc)
    assert _grouped(eng, b) == want
    # n == 0: accept
    assert eng.verify_multiple_grouped(None, b"", b"", None, b"", [0], [], []) == (True, -1)


def _edge_grouped():
    """The edge sets of the locate tests, with their messages drawn from a pool of four so that sets share groups."""
    rnd = random.Random(0x10CA7E)
    sk = [rnd.randrange(1, O.r) for _ in range(12)]
    pk = [O.sk_to_pk(s) for s in sk]
    pool = [b"grouped %d" % k + bytes(20) for k in range(4)]
    msg = [pool[j % 4] for j in range(24)]
    D = O.hash_to_curve_g2(b"cancelling difference")
    sets = []

    def signed(keys, m):
        return O.aggregate_signatures([O.sign(sk[k], m) for k in keys])

    for j, keys in enumerate(([0], [1, 2], [3, 4, 5], [6, 7], [8], [9, 10, 11])):
        sets.append((signed(keys, msg[j]), [pk[k] for k in keys], msg[j], True))
    sets.append((signed([0, 1], msg[6]), [pk[0], pk[1]], msg[6][:-1] + b"\x01", False))        # tampered message: its own group
    sets.append((sets[0][0], [pk[0]], msg[7], False))                                           # another message's signature
    sets.append((signed([2, 3], msg[8]), [pk[2], pk[4]], msg[8], False))                        # wrong key set
    sets.append((O.aggregate_signatures([O.sign(sk[5], msg[9])] * 2 + [O.sign(sk[6], msg[9])]), [pk[5], pk[5], pk[6]], msg[9], True))
    sets.append((signed([5, 6], msg[10]), [pk[5], pk[5], pk[6]], msg[10], False))
    sets.append((O.map_to_curve_g2((5, 7)), [pk[7]], msg[11], False))                          # non-subgroup signature
    sets.append((None, [pk[8], O.g1_neg(pk[8])], msg[12], True))
    sets.append((None, [pk[9]], msg[13], False))
    sets.append((signed([10], msg[14]), [pk[10], O.g1_neg(pk[10])], msg[14], False))
    sets.append((signed([11], msg[15]), [], msg[15], False))
    sets.append((None, [], msg[16], True))
    sets.append((O.g2_add(signed([0, 3], msg[17]), D), [pk[0], pk[3]], msg[17], False))
    sets.append((O.g2_add(signed([1, 4], msg[18]), O.g2_neg(D)), [pk[1], pk[4]], msg[18], False))
    for j, keys in zip(range(19, 24), ([2], [3, 6], [7, 8, 9], [10], [11, 0])):
        sets.append((signed(keys, msg[j]), [pk[k] for k in keys], msg[j], True))
    msgs = []
    for _, _, m, _ in sets:
        if m not in msgs:
            msgs.append(m)
    rs = random.Random(7)
    return {"sigs": u8(b"".join(g2w(s) for s, _, _, _ in sets)), "pks": u8(b"".join(g1w(P) for _, ks, _, _ in sets for P in ks)),
            "pk_off": _offs([[0] * len(ks) for _, ks, _, _ in sets]), "msgs": msgs,
            "mi": np.array([msgs.index(m) for _, _, m, _ in sets], dtype=np.uint32),
            "scalars": np.array([rs.randrange(1, 1 << 63) for _ in sets], dtype=np.uint64), "want": [w for _, _, _, w in sets]}


def test_locate_after_grouped(eng):
    b = _edge_grouped()
    n = len(b["want"])
    assert len(b["msgs"]) == 5 and max(np.bincount(b["mi"])) >= 5
    ok, fb, _ = _same(eng, b)
    assert not ok and fb == 11
    after_expanded = eng.verify_multiple_locate(n)                # _same ran the expanded call last
    _grouped(eng, b)
    after_grouped = eng.verify_multiple_locate(n)
    assert after_grouped.tolist() == after_expanded.tolist() == b["want"]
    for kern in (1, 3):                                           # both finishing kernels read H's pair by message index
        eng.set_item_kernel(kern)
        try:
            assert eng.verify_multiple_locate(n).tolist() == b["want"]
        finally:
            eng.set_item_kernel(0)
    # state rules: a wrong n, another call in between, and an accepting grouped call
    with pytest.raises(RuntimeError, match="BadArgument"):
        eng.verify_multiple_locate(n - 1)
    eng.hash_to_g2([b"x"])
    with pytest.raises(RuntimeError, match="BadArgument"):
        eng.verify_multiple_locate(n)
    good = [j for j in range(n) if b["want"][j]]
    sub = {"sigs": np.concatenate([b["sigs"][192 * j:192 * (j + 1)] for j in good]),
           "pks": np.concatenate([b["pks"][96 * int(b["pk_off"][j]):96 * int(b["pk_off"][j + 1])] for j in good]),
           "pk_off": _offs([[0] * int(b["pk_off"][j + 1] - b["pk_off"][j]) for j in good]), "msgs": b["msgs"], "mi": b["mi"][good],
           "scalars": b["scalars"][good]}
    ok, _, _ = _grouped(eng, sub)
    assert ok
    before = eng.launches
    assert eng.verify_multiple_locate(len(good)).all() and eng.launches == before


def test_python_extension(eng):
    import milagro_bls_b200 as mb
    rnd = random.Random(0xE87)
    sk = [rnd.randrange(1, O.r) for _ in range(6)]
    pool = [b"ext root", b"ext data", b"ext other"]
    sets_ok = []
    for j in range(9):
        m = pool[j % 3] if j < 6 else b"ext unique %d" % j
        sets_ok.append((mb.AggregateSignature(g2w(O.sign(sk[j % 6], m))), mb.AggregatePublicKey(g1w(O.sk_to_pk(sk[j % 6]))), m))
    ns = mb.AggregateSignature(g2w(O.map_to_curve_g2((5, 7))))
    cases = {"valid": sets_ok,
             "swapped": [sets_ok[0], (sets_ok[2][0], sets_ok[1][1], sets_ok[1][2])] + sets_ok[2:],
             "non-subgroup": sets_ok[:4] + [(ns, sets_ok[4][1], sets_ok[4][2])] + sets_ok[5:],
             "unique": sets_ok[6:], "empty": []}
    for name, sets in cases.items():
        r1, r2 = mb.SeededRng(b"grouped " + name.encode()), mb.SeededRng(b"grouped " + name.encode())
        got = mb.AggregateSignature.verify_multiple_aggregate_signatures_grouped(r1, sets, engine=eng)
        want = mb.AggregateSignature.verify_multiple_aggregate_signatures(r2, sets, engine=eng)
        assert got == want == (name in ("valid", "unique", "empty")), name
        assert r1.fill(16) == r2.fill(16), name
