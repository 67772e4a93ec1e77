"""b3_verify_multiple_locate: the per-set verdicts of a rejected verify_multiple batch, read from what the batch call left on the
device.  valid[j] must be exactly "set j alone passes verify_multiple_aggregate_signatures" (M/src/aggregates.rs:261-316):

  * edge sets (valid, tampered, swapped, wrong keys, duplicate keys, non-subgroup signature, the infinities, an empty key range
    and a cancelling pair whose unweighted sum verifies) against the C oracle, the Python oracle for the infinity cases, and the
    library's own verify_multiple over the set alone;
  * every whole entry (byte keys with and without pk_off, _checked, _indexed with and without pk_off, _dev, _indexed_dev),
    latency modes, finishing kernels and serial / overlapped stages give the same verdicts;
  * sizes around the signature-MSM switch (512 sets) and the CTA / lane-pair switch (2048), bad sets first and last;
  * the C4 batch (8192 sets x 128 keys);
  * the state rules (enabled only by a whole call, repeatable, leaves the next call unchanged) and the Python extension.
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


@pytest.fixture(scope="module")
def edge():
    return _edge_sets()


def _edge_sets():
    """About 24 sets (signature point, key points, message, expected verdict, whether an infinity is involved)."""
    rnd = random.Random(0x10CA7E)
    sk = [rnd.randrange(1, O.r) for _ in range(12)]
    pk = [O.sk_to_pk(s) for s in sk]
    msg = [b"locate %02d" % j + bytes(20) for j in range(24)]
    D = O.hash_to_curve_g2(b"cancelling difference")
    sets = []

    def signed(keys, m):
        return O.aggregate_signatures([O.sign(sk[k], m) for k in keys])

    for j, keys in enumerate(([0], [1, 2], [3, 4, 5], [6, 7], [8], [9, 10, 11])):          # 0-5: valid
        sets.append((signed(keys, msg[j]), [pk[k] for k in keys], msg[j], True, False))
    sets.append((signed([0, 1], msg[6]), [pk[0], pk[1]], msg[6][:-1] + b"\x01", False, False))   # 6: tampered message
    sets.append((sets[0][0], [pk[0]], msg[7], False, False))                                     # 7: another message's signature
    sets.append((signed([2, 3], msg[8]), [pk[2], pk[4]], msg[8], False, False))                  # 8: wrong key set
    sets.append((O.aggregate_signatures([O.sign(sk[5], msg[9])] * 2 + [O.sign(sk[6], msg[9])]),  # 9: duplicate key, counted twice
                 [pk[5], pk[5], pk[6]], msg[9], True, False))
    sets.append((signed([5, 6], msg[10]), [pk[5], pk[5], pk[6]], msg[10], False, False))        # 10: duplicate key, signed once
    ns = O.map_to_curve_g2((5, 7))
    assert O.g2_is_on_curve(ns) and not O.subgroup_check_g2(ns)
    sets.append((ns, [pk[7]], msg[11], False, False))                                            # 11: on-curve non-subgroup signature
    sets.append((None, [pk[8], O.g1_neg(pk[8])], msg[12], True, True))                          # 12: sig = inf, apk = inf
    sets.append((None, [pk[9]], msg[13], False, True))                                           # 13: sig = inf, real apk
    sets.append((signed([10], msg[14]), [pk[10], O.g1_neg(pk[10])], msg[14], False, True))      # 14: pk and -pk, real sig
    sets.append((signed([11], msg[15]), [], msg[15], False, True))                               # 15: empty key range, real sig
    sets.append((None, [], msg[16], True, True))                                                 # 16: empty key range, sig = inf
    sa, sb = signed([0, 3], msg[17]), signed([1, 4], msg[18])
    sets.append((O.g2_add(sa, D), [pk[0], pk[3]], msg[17], False, False))                        # 17, 18: cancelling pair
    sets.append((O.g2_add(sb, O.g2_neg(D)), [pk[1], pk[4]], msg[18], False, False))
    for j, keys in zip(range(19, 24), ([2], [3, 6], [7, 8, 9], [10], [11, 0])):                  # 19-23: valid
        sets.append((signed(keys, msg[j]), [pk[k] for k in keys], msg[j], True, False))
    n = len(sets)
    sigs = b"".join(g2w(s) for s, _, _, _, _ in sets)
    pks = b"".join(g1w(P) for _, ks, _, _, _ in sets for P in ks)
    pk_off = np.zeros(n + 1, dtype=np.uint32)
    pk_off[1:] = np.cumsum([len(ks) for _, ks, _, _, _ in sets])
    apks = b"".join(g1w(_g1_sum(ks)) for _, ks, _, _, _ in sets)
    msgs = [m for _, _, m, _, _ in sets]
    rs = random.Random(7)
    scalars = np.array([rs.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    # the key table holds every distinct key once; idx names them per set
    table_pts, idx = [], []
    for _, ks, _, _, _ in sets:
        for P in ks:
            w = g1w(P)
            if w not in table_pts:
                table_pts.append(w)
            idx.append(table_pts.index(w))
    return {"sets": sets, "n": n, "sigs": u8(sigs), "pks": u8(pks), "pk_off": pk_off, "apks": u8(apks), "msgs": msgs,
            "blob": b"".join(msgs), "moff": np.array([0] + list(np.cumsum([len(m) for m in msgs])), dtype=np.uint32),
            "scalars": scalars, "table": b"".join(table_pts), "idx": np.array(idx, dtype=np.uint32),
            "want": np.array([w for _, _, _, w, _ in sets])}


def _g1_sum(ks):
    acc = None
    for P in ks:
        acc = O.g1_add(acc, P)
    return acc


def _set_args(e, j):
    """The arguments of verify_multiple over set j alone (keys through pk_off)."""
    a, b = int(e["pk_off"][j]), int(e["pk_off"][j + 1])
    return (e["sigs"][192 * j:192 * (j + 1)], e["pks"][96 * a:96 * b], np.array([0, b - a], dtype=np.uint32), e["msgs"][j],
            np.array([0, len(e["msgs"][j])], dtype=np.uint32), e["scalars"][j:j + 1])


def test_edge_sets_against_oracles(eng, edge):
    e = edge
    ok, fb = eng.verify_multiple(e["sigs"], e["pks"], e["pk_off"], e["blob"], e["moff"], e["scalars"])
    assert not ok and fb == 11
    valid = eng.verify_multiple_locate(e["n"])
    assert valid.tolist() == e["want"].tolist()
    for j, (sig, ks, m, want, has_inf) in enumerate(e["sets"]):
        args = _set_args(e, j)
        ok_c, _ = c_oracle.verify_multiple(*args)
        assert ok_c == want, j
        if has_inf:
            assert O.verify_multiple_aggregate_signatures(O.SeededRng(b"%d" % j).fill, [(sig, _g1_sum(ks), m)]) == want, j
        assert eng.verify_multiple(*args)[0] == want, j
    # the cancelling pair: their unweighted sum verifies, yet each set is invalid
    s17, s18 = e["sets"][17], e["sets"][18]
    assert O.aggregate_verify(O.g2_add(s17[0], s18[0]), [s17[2], s18[2]], [_g1_sum(s17[1]), _g1_sum(s18[1])])


def _dev(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a).view(np.uint8).reshape(-1).copy()).to(torch.device("cuda", 0))


def test_every_whole_entry_gives_the_same_verdicts(eng, edge):
    import milagro_bls_b200 as mb
    e = edge
    n, want = e["n"], e["want"].tolist()
    args = (e["blob"], e["moff"], e["scalars"])
    # byte keys through pk_off and as one aggregate key per set
    eng.verify_multiple(e["sigs"], e["pks"], e["pk_off"], *args)
    assert eng.verify_multiple_locate(n).tolist() == want
    eng.verify_multiple(e["sigs"], e["apks"], None, *args)
    assert eng.verify_multiple_locate(n).tolist() == want
    # _checked after a passing precheck: the non-subgroup signature fails the precheck, so the batch without it
    keep = [j for j in range(n) if j != 11]
    sub_sigs = np.concatenate([e["sigs"][192 * j:192 * (j + 1)] for j in keep])
    sub_apks = np.concatenate([e["apks"][96 * j:96 * (j + 1)] for j in keep])
    sub_msgs = [e["msgs"][j] for j in keep]
    sub_moff = np.array([0] + list(np.cumsum([len(m) for m in sub_msgs])), dtype=np.uint32)
    assert eng.sig_precheck(sub_sigs) == -1
    eng.verify_multiple_checked(sub_apks, None, b"".join(sub_msgs), sub_moff, e["scalars"][keep])
    assert eng.verify_multiple_locate(len(keep)).tolist() == [want[j] for j in keep]
    # key table: indices through pk_off, and one entry per set (sets whose aggregate key is not infinity)
    tbl = mb.KeyTable(eng)
    _, st = tbl.append(u8(e["table"]), compressed=False, validate=True)
    assert not st.any()
    eng.verify_multiple_indexed(tbl, e["sigs"], e["idx"], e["pk_off"], *args)
    assert eng.verify_multiple_locate(n).tolist() == want
    fin = [j for j in range(n) if e["apks"][96 * j] & 0x40 == 0]
    first, st = tbl.append(np.concatenate([e["apks"][96 * j:96 * (j + 1)] for j in fin]), compressed=False, validate=True)
    assert not st.any()
    fin_msgs = [e["msgs"][j] for j in fin]
    eng.verify_multiple_indexed(tbl, np.concatenate([e["sigs"][192 * j:192 * (j + 1)] for j in fin]),
                                np.arange(first, first + len(fin), dtype=np.uint32), None, b"".join(fin_msgs),
                                np.array([0] + list(np.cumsum([len(m) for m in fin_msgs])), dtype=np.uint32), e["scalars"][fin])
    assert eng.verify_multiple_locate(len(fin)).tolist() == [want[j] for j in fin]
    # inputs resident in HBM
    d = [_dev(a) for a in (e["sigs"], e["pks"], e["pk_off"], u8(e["blob"]), e["moff"], e["scalars"], e["idx"])]
    ok, fb = eng.verify_multiple_dev(None, d[0].data_ptr(), d[1].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), d[4].data_ptr(),
                                     d[5].data_ptr(), n)
    assert not ok and fb == 11
    assert eng.verify_multiple_locate(n).tolist() == want
    eng.verify_multiple_dev(tbl, d[0].data_ptr(), d[6].data_ptr(), d[2].data_ptr(), d[3].data_ptr(), d[4].data_ptr(), d[5].data_ptr(), n)
    assert eng.verify_multiple_locate(n).tolist() == want
    # latency modes, finishing kernels, serial / overlapped stages
    try:
        for mode in (1, 2):
            for kern in (1, 3):
                for serial in (True, False):
                    eng.set_latency_mode(mode)
                    eng.set_item_kernel(kern)
                    eng.set_serial(serial)
                    eng.verify_multiple(e["sigs"], e["pks"], e["pk_off"], *args)
                    assert eng.verify_multiple_locate(n).tolist() == want, (mode, kern, serial)
    finally:
        eng.set_latency_mode(0)
        eng.set_item_kernel(0)
        eng.set_serial(False)


def _synth(eng, n, nk, seed):
    """n valid sets of nk keys each (signing-side work on the library's input helpers)."""
    rnd = random.Random(seed)
    pool_n = max(4 * nk, 64)
    sks = [rnd.randrange(1, O.r) for _ in range(pool_n)]
    pool = eng.g1_mul_gen(sks)
    rs = np.random.RandomState(seed & 0xffff)
    idx = np.stack([rs.choice(pool_n, size=nk, replace=False) for _ in range(n)]).astype(np.uint32)
    msgs = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    msgs[:, :4] = np.arange(n, dtype=">u4").view(np.uint8).reshape(n, 4)
    agg_sk = [sum(sks[i] for i in row) % O.r for row in idx]
    H = eng.hash_to_g2([m.tobytes() for m in msgs])
    sigs = eng.g2_mul(H.reshape(-1), agg_sk)
    scalars = np.array([rnd.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    return {"n": n, "nk": nk, "pool": pool, "idx": idx, "pks": np.ascontiguousarray(pool[idx.reshape(-1)]).reshape(-1),
            "pk_off": np.arange(0, n * nk + 1, nk, dtype=np.uint32), "msgs": msgs, "moff": np.arange(0, 32 * n + 1, 32, dtype=np.uint32),
            "sigs": np.ascontiguousarray(sigs).reshape(-1), "scalars": scalars}


@pytest.mark.parametrize("n", [1, 2, 511, 512, 513, 2047, 2048])
def test_sizes_at_the_boundaries(eng, n):
    b = _synth(eng, n, 4, 0x5E7 + n)
    tam = b["msgs"].copy()
    bad = sorted({0, n - 1})
    for j in bad:
        tam[j, 17] ^= 0x10
    ok, fb = eng.verify_multiple(b["sigs"], b["pks"], b["pk_off"], tam.reshape(-1), b["moff"], b["scalars"])
    assert not ok and fb == -1
    want = np.ones(n, dtype=bool)
    want[bad] = False
    assert np.array_equal(eng.verify_multiple_locate(n), want)
    # the valid batch: all ones, nothing launched
    ok, _ = eng.verify_multiple(b["sigs"], b["pks"], b["pk_off"], b["msgs"].reshape(-1), b["moff"], b["scalars"])
    assert ok
    before = eng.launches
    assert eng.verify_multiple_locate(n).all() and eng.launches == before


@pytest.fixture(scope="module")
def c4(eng):
    """The C4 batch: 8192 sets x 128 keys drawn from a pool of 4096 validators."""
    rnd = random.Random(0xC4)
    n, nk, pool_n = 8192, 128, 4096
    sks = [rnd.randrange(1, O.r) for _ in range(pool_n)]
    pool = eng.g1_mul_gen(sks)
    rs = np.random.RandomState(4)
    idx = np.stack([rs.choice(pool_n, size=nk, replace=False) for _ in range(n)]).astype(np.uint32)
    msgs = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    msgs[:, :4] = np.arange(n, dtype=">u4").view(np.uint8).reshape(n, 4)
    agg_sk = [sum(sks[i] for i in row) % O.r for row in idx]
    H = eng.hash_to_g2([m.tobytes() for m in msgs])
    sigs = eng.g2_mul(H.reshape(-1), agg_sk)
    assert sigs[5].tobytes() == g2w(O.g2_mul(O.hash_to_curve_g2(msgs[5].tobytes()), agg_sk[5]))
    scalars = np.array([rnd.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    return {"n": n, "nk": nk, "pool": pool, "idx": idx, "pks": np.ascontiguousarray(pool[idx.reshape(-1)]).reshape(-1),
            "pk_off": np.arange(0, n * nk + 1, nk, dtype=np.uint32), "msgs": msgs, "moff": np.arange(0, 32 * n + 1, 32, dtype=np.uint32),
            "sigs": np.ascontiguousarray(sigs).reshape(-1), "scalars": scalars}


def test_c4_exact_verdict_vectors(eng, c4):
    n = c4["n"]
    ns = np.frombuffer(g2w(O.map_to_curve_g2((5, 7))), dtype=np.uint8)
    spread = [0, 1, 77, 511, 512, 1000, 2047, 2048, 3333, 4095, 4096, 5003, 6001, 7000, 8190, 8191]
    cases = [({5003}, None), (set(spread), None), (set(range(n)), None), ({12}, 7000)]
    for tampered, nonsub in cases:
        msgs, sigs = c4["msgs"].copy(), c4["sigs"]
        for j in tampered:
            msgs[j, 9] ^= 0x40
        if nonsub is not None:
            sigs = sigs.copy()
            sigs[192 * nonsub:192 * (nonsub + 1)] = ns
        ok, fb = eng.verify_multiple(sigs, c4["pks"], c4["pk_off"], msgs.reshape(-1), c4["moff"], c4["scalars"])
        assert not ok and fb == (-1 if nonsub is None else nonsub)
        want = np.ones(n, dtype=bool)
        want[sorted(tampered)] = False
        if nonsub is not None:
            want[nonsub] = False
        assert np.array_equal(eng.verify_multiple_locate(n), want), sorted(tampered)


def test_state_rules(eng):
    import torch
    b = _synth(eng, 40, 3, 0x57A7E)
    tam = b["msgs"].copy()
    tam[21, 3] ^= 1
    args = (b["sigs"], b["pks"], b["pk_off"], tam.reshape(-1), b["moff"], b["scalars"])
    want = np.ones(40, dtype=bool)
    want[21] = False
    # enabled by a whole call only, for its n only
    ok, fb, gt = eng.verify_multiple(*args, want_gt=True)
    assert not ok
    with pytest.raises(RuntimeError, match="BadArgument"):
        eng.verify_multiple_locate(39)
    v1 = eng.verify_multiple_locate(40)
    v2 = eng.verify_multiple_locate(40)
    assert np.array_equal(v1, want) and np.array_equal(v2, want)
    # the next call is unchanged by locate
    assert eng.verify_multiple(*args, want_gt=True) == (ok, fb, gt)
    assert np.array_equal(eng.verify_multiple_locate(40), want)
    # any other call ends the window
    others = [lambda: eng.hash_to_g2([b"x"]),
              lambda: eng.verify_batch(1, b["sigs"][:192], b["pks"][:96 * 3], [0, 3], [b["msgs"][0].tobytes()]),
              lambda: eng.sig_precheck(b["sigs"]),
              lambda: eng.verify_multiple_partial(*args, 0, part.data_ptr())]
    part = torch.zeros(592, dtype=torch.uint8, device="cuda")
    import milagro_bls_b200 as mb
    tbl = mb.KeyTable(eng)
    others.append(lambda: tbl.append(b["pool"][:2].reshape(-1), compressed=False))
    for other in others:
        eng.verify_multiple(*args)
        other()
        with pytest.raises(RuntimeError, match="BadArgument"):
            eng.verify_multiple_locate(40)
    # a call that raised (scalar 0) does not enable it either
    sc0 = b["scalars"].copy()
    sc0[3] = 0
    with pytest.raises(RuntimeError):
        eng.verify_multiple(*args[:5], sc0)
    with pytest.raises(RuntimeError, match="BadArgument"):
        eng.verify_multiple_locate(40)


def test_python_extension(eng, edge):
    import milagro_bls_b200 as mb
    e = edge
    sets = [(mb.AggregateSignature(g2w(s)), mb.AggregatePublicKey(g1w(_g1_sum(ks))), m) for s, ks, m, _, _ in e["sets"]]
    rng = mb.SeededRng(b"per set")
    got = mb.AggregateSignature.verify_multiple_aggregate_signatures_per_set(rng, sets, engine=eng)
    assert got == e["want"].tolist()
    ref = mb.SeededRng(b"per set")
    for _ in sets:
        mb.draw_scalar(ref)
    assert rng.fill(16) == ref.fill(16)                   # exactly one scalar per set was drawn
    good = [sets[j] for j in range(len(sets)) if e["want"][j]]
    assert mb.AggregateSignature.verify_multiple_aggregate_signatures_per_set(mb.SeededRng(b"g"), good, engine=eng) == [True] * len(good)
    assert mb.AggregateSignature.verify_multiple_aggregate_signatures_per_set(mb.SeededRng(b"g"), [], engine=eng) == []
    broken = list(sets)
    broken[4] = (mb.AggregateSignature(bytes([0x80]) + bytes(191)), broken[4][1], broken[4][2])
    with pytest.raises(mb.AmclError):
        mb.AggregateSignature.verify_multiple_aggregate_signatures_per_set(mb.SeededRng(b"b"), broken, engine=eng)
