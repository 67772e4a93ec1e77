"""The signature sum S = sum_j [c_j] sig_j of verify_multiple by the bucket method (from 512 sets: digit sort per 8-bit window,
running-sum walk over the sorted lists, csrc/kernels.cuh k_msm_*), under scalar distributions that stress the buckets:
every set in one bucket, zero digits, the extreme 64-bit values (the top window has digits up to 255) and random scalars.
Up to 640 sets a rejecting batch's GT is compared byte for byte with the C oracle; above, a wrong S would reject a valid
batch, so every valid batch must accept and the same batch with one tampered message must reject."""
import random

import numpy as np
import pytest

from oracle import bls_oracle as O

pytestmark = pytest.mark.gpu
ORACLE_MAX = 640
KINDS = ["equal", "zero_digits", "extremes", "random"]


@pytest.fixture(scope="module")
def eng():
    import __graft_entry__ as g
    g.build_cuda()
    import milagro_bls_b200 as mb
    e = mb.Engine(0)
    mb.set_default_engine(e)
    return e


_BATCHES = {}


def _batch(eng, n):
    """n valid single-key sets: sig_j = [sk_j] H(m_j), pk_j = [sk_j] G1 (synthesised on the GPU)."""
    if n not in _BATCHES:
        rnd = random.Random(1000 + n)
        sks = [rnd.randrange(1, O.r) for _ in range(n)]
        pk = eng.g1_mul_gen(sks)
        msgs = [rnd.getrandbits(256).to_bytes(32, "big") for _ in range(n)]
        sig = eng.g2_mul(eng.hash_to_g2(msgs).reshape(-1), sks)
        _BATCHES[n] = (sig.reshape(-1), pk.reshape(-1), msgs, list(range(0, 32 * n + 1, 32)))
    return _BATCHES[n]


def _scalars(kind, n):
    rnd = random.Random(f"{kind}-{n}")
    if kind == "equal":
        return np.full(n, 0x9e3779b97f4a7c15, dtype=np.uint64)                   # every set in one bucket of each window
    if kind == "zero_digits":
        vals = [1, 1 << 56, 0x0100, 0x0100000000000001, 0xff00ff00ff00ff00, 0x00000000ffffffff]
        return np.array([vals[j % len(vals)] for j in range(n)], dtype=np.uint64)
    if kind == "extremes":
        vals = [(1 << 63) - 1, 1 << 63, (1 << 64) - 1]
        return np.array([vals[j % 3] for j in range(n)], dtype=np.uint64)
    return np.array([rnd.getrandbits(64) | 1 for _ in range(n)], dtype=np.uint64)


@pytest.mark.parametrize("kind", KINDS)
@pytest.mark.parametrize("n", [512, 513, 8191, 8192, 8193, 32768])
def test_msm_scalar_distributions(eng, n, kind):
    from oracle import c_oracle
    sig, pk, msgs, moff = _batch(eng, n)
    sc = _scalars(kind, n)
    ok, fb, gt = eng.verify_multiple(sig, pk, None, b"".join(msgs), moff, sc, want_gt=True)
    assert ok and fb == -1 and gt == O.f12_to_bytes(O.F12_ONE)
    bad = n // 3
    tampered = list(msgs); tampered[bad] = b"tampered" + msgs[bad][8:]
    ok, fb, gt = eng.verify_multiple(sig, pk, None, b"".join(tampered), moff, sc, want_gt=True)
    assert not ok and fb == -1 and gt != O.f12_to_bytes(O.F12_ONE)
    if n <= ORACLE_MAX:
        ok_c, gt_c = c_oracle.verify_multiple(sig, pk, None, b"".join(tampered), moff, sc)
        assert not ok_c and gt == gt_c


@pytest.mark.parametrize("kind", ["equal", "random"])
def test_msm_partial_is_deterministic(eng, kind):
    """The Miller product (before the final exponentiation) depends on the coordinates of the window sums: two identical
    calls must leave byte-identical 592-byte partial records."""
    import torch
    n = 8192
    sig, pk, msgs, moff = _batch(eng, n)
    dev = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dtype=dt)).cuda()
    d_sig, d_pk = dev(sig, np.uint8), dev(pk, np.uint8)
    d_msg, d_moff = dev(np.frombuffer(b"".join(msgs), dtype=np.uint8), np.uint8), dev(moff, np.uint32)
    d_sc = dev(_scalars(kind, n).view(np.int64), np.int64)
    parts = [torch.zeros(592, dtype=torch.uint8, device="cuda:0") for _ in range(2)]
    torch.cuda.synchronize()
    for p in parts:
        eng.verify_multiple_partial_dev(d_sig.data_ptr(), d_pk.data_ptr(), None, d_msg.data_ptr(), d_moff.data_ptr(), d_sc.data_ptr(),
                                        n, 0, p.data_ptr())
        torch.cuda.synchronize()
    assert torch.equal(parts[0], parts[1])
    assert eng.combine_partials_dev(parts[0].data_ptr(), 1) == (True, -1)


def test_msm_one_bucket_costs_no_more_than_random(eng):
    """All sets in one bucket of every window is the same number of walk events as random scalars: with the stages
    serialised, its MSM stage must take no more than twice the random one (median of 5 calls each, C4 size)."""
    n = 8192
    sig, pk, msgs, moff = _batch(eng, n)
    blob = b"".join(msgs)
    ms = {}
    eng.set_serial(True)
    try:
        for kind in ("random", "equal"):
            sc = _scalars(kind, n)
            t = []
            for _ in range(6):
                assert eng.verify_multiple(sig, pk, None, blob, moff, sc)[0]
                t.append(eng.stage_ms()["g2_scalar_mul_sum"])
            ms[kind] = float(np.median(t[1:]))
    finally:
        eng.set_serial(False)
    assert ms["equal"] <= 2 * ms["random"], ms
