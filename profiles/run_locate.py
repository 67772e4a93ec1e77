"""Timing of b3_verify_multiple_locate against what a caller can do without it (b3_verify_batch over the same sets).

Shape: 128 keys per set, named by index into a device-resident key table (the b3_verify_multiple_indexed path); n in
{256, 8192, 32768}, each with 1 bad set (a tampered message), 16 spread bad sets and every set bad.  Per case, after two
warm-up rounds, the median of `reps` rounds of:
  batch   b3_verify_multiple_indexed (host pointers), which rejects
  locate  b3_verify_multiple_locate on the same context
  batch_items  b3_verify_batch(B3_ITEM_FAST_AGGREGATE) over the same sets with 96-byte keys: what a caller has to run today
Each call ends in a device synchronise; `host` is a host clock around it, `dev` the library's own event time of the call
(b3_ctx_last_kernel_ms(0): from its first enqueued work, copies included, to its last kernel), `fin` locate's finishing
kernel alone.  The verdict vectors of locate and of verify_batch are checked against the tampered set list in every round.
The card's name and power limit are read in the same run.

usage: python profiles/run_locate.py [out.txt] [reps]"""
import os
import random
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import milagro_bls_b200 as mb  # noqa: E402
from milagro_bls_b200 import _lib  # noqa: E402

R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
KEYS, POOL = 128, 4096


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                      # the device name still comes from torch
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name(0)}; nvidia-smi: {q}"


def synth(eng, n, pool, sks, rnd):
    rs = np.random.RandomState(n)
    idx = np.stack([rs.choice(POOL, size=KEYS, replace=False) for _ in range(n)]).astype(np.uint32)
    msgs = rs.randint(0, 256, size=(n, 32), dtype=np.uint8)
    msgs[:, :4] = np.arange(n, dtype=">u4").view(np.uint8).reshape(n, 4)
    agg_sk = [sum(sks[i] for i in row) % R for row in idx]
    H = eng.hash_to_g2([m.tobytes() for m in msgs])
    sigs = np.ascontiguousarray(eng.g2_mul(H.reshape(-1), agg_sk)).reshape(-1)
    scalars = np.array([rnd.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    return idx, msgs, sigs, scalars


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    eng = mb.Engine(0)
    say(f"# b3_verify_multiple_locate vs b3_verify_batch, {KEYS} keys per set (key table indices), median of {reps} after 2 warm-up rounds")
    say(f"# card: {card()}")
    rnd = random.Random(0x10CA7E)
    sks = [rnd.randrange(1, R) for _ in range(POOL)]
    pool = eng.g1_mul_gen(sks)
    tbl = mb.KeyTable(eng)
    _, st = tbl.append(pool.reshape(-1), compressed=False, validate=True)
    assert not st.any()
    say(f"{'n':>6} {'bad':>6} | {'batch host':>10} {'dev':>8} | {'locate host':>11} {'dev':>8} {'fin':>8} | "
        f"{'verify_batch host':>17} {'dev':>8} | {'locate / verify_batch':>21}")
    for n in (256, 8192, 32768):
        idx, msgs, sigs, scalars = synth(eng, n, pool, sks, rnd)
        kidx = idx.reshape(-1)
        koff = np.arange(0, n * KEYS + 1, KEYS, dtype=np.uint32)
        moff = np.arange(0, 32 * n + 1, 32, dtype=np.uint32)
        pks = np.ascontiguousarray(pool[kidx]).reshape(-1)
        spread = sorted({0, n - 1} | set(np.linspace(0, n - 1, 16).astype(int).tolist()))[:16]
        for label, bad in (("1", [n // 2 + 3]), ("16", spread), ("all", list(range(n)))):
            tam = msgs.copy()
            tam[bad, 9] ^= 0x40
            blob = tam.reshape(-1)
            msg_list = [m.tobytes() for m in tam]
            want = np.ones(n, dtype=bool)
            want[bad] = False
            t = {"batch": [], "batch_dev": [], "loc": [], "loc_dev": [], "fin": [], "vb": [], "vb_dev": []}
            for r in range(reps + 2):
                t0 = time.perf_counter()
                ok, fb = eng.verify_multiple_indexed(tbl, sigs, kidx, koff, blob, moff, scalars)
                t1 = time.perf_counter()
                bdev = eng.last_kernel_ms(0)
                assert not ok and fb == -1
                valid = eng.verify_multiple_locate(n)
                t2 = time.perf_counter()
                ldev, lfin = eng.last_kernel_ms(0), eng.last_kernel_ms(1)
                assert np.array_equal(valid, want)
                t3 = time.perf_counter()
                acc, st = eng.verify_batch(_lib.ITEM_FAST_AGGREGATE, sigs, pks, koff, msg_list)
                t4 = time.perf_counter()
                vdev = eng.last_kernel_ms(0)
                assert np.array_equal(acc, want) and not st.any()
                if r >= 2:
                    for k, v in (("batch", (t1 - t0) * 1e3), ("batch_dev", bdev), ("loc", (t2 - t1) * 1e3), ("loc_dev", ldev), ("fin", lfin),
                                 ("vb", (t4 - t3) * 1e3), ("vb_dev", vdev)):
                        t[k].append(v)
            m = {k: float(np.median(v)) for k, v in t.items()}
            say(f"{n:>6} {label:>6} | {m['batch']:>10.2f} {m['batch_dev']:>8.2f} | {m['loc']:>11.2f} {m['loc_dev']:>8.2f} {m['fin']:>8.2f} | "
                f"{m['vb']:>17.2f} {m['vb_dev']:>8.2f} | {m['loc'] / m['vb']:>21.3f}")
    say("# times in ms; 'locate / verify_batch' = ratio of the host-clock medians")
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
