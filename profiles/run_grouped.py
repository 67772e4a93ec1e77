"""Timing of b3_verify_multiple_grouped against the ungrouped call on the expanded inputs (every set's message written out).

Shapes (valid batches, one call in flight on the device):
  512 x 1 key, 1 message               (a sync-committee slot: 96-byte keys)
  8192 x 1 key over 64 messages        (unaggregated attestations of 64 committees: 96-byte keys)
  8192 x 128 table keys over 64 messages
  8192 x 128 table keys, all distinct  (nothing shared: the cost of the sort and the segmented sum)
Per shape, after two warm-up rounds, the median of `reps` rounds, each running the grouped and the expanded call back to back
(alternating which goes first).  Each call ends in a device synchronise; `host` is a host clock around it, `dev` the library's
own event time (b3_ctx_last_kernel_ms(0)).  Accept bits and GT bytes of the two calls are compared in every round.  Then one
serial round of each (stages one after another on one stream) gives the per-stage device times.  The card's name and power
limit are read in the same run.

usage: python profiles/run_grouped.py [out.txt] [reps]"""
import os
import random
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import milagro_bls_b200 as mb  # noqa: E402

R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
POOL = 4096


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:                      # the device name still comes from torch
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name(0)}; nvidia-smi: {q}"


def offs(chunks):
    return np.array([0] + list(np.cumsum([len(c) for c in chunks])), dtype=np.uint32)


def synth(eng, pool, sks, n, nk, n_msgs, seed):
    rs = np.random.RandomState(seed)
    rnd = random.Random(seed)
    idx = np.stack([rs.choice(POOL, size=nk, replace=False) for _ in range(n)]).astype(np.uint32)
    msgs = rs.randint(0, 256, size=(n_msgs, 32), dtype=np.uint8)
    msgs[:, :4] = np.arange(n_msgs, dtype=">u4").view(np.uint8).reshape(n_msgs, 4)
    mi = np.arange(n, dtype=np.uint32) if n_msgs == n else rs.randint(0, n_msgs, size=n).astype(np.uint32)
    agg_sk = [sum(sks[i] for i in row) % R for row in idx]
    H = eng.hash_to_g2([m.tobytes() for m in msgs])
    sigs = np.ascontiguousarray(eng.g2_mul(np.ascontiguousarray(H[mi]).reshape(-1), agg_sk)).reshape(-1)
    scalars = np.array([rnd.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    msg_list = [m.tobytes() for m in msgs]
    ex = [msg_list[k] for k in mi]
    return {"idx": idx, "mi": mi, "msgs": msg_list, "ex": ex, "sigs": sigs, "scalars": scalars,
            "pk_off": np.arange(0, n * nk + 1, nk, dtype=np.uint32)}


def main():
    out_path = sys.argv[1] if len(sys.argv) > 1 else None
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 7
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    eng = mb.Engine(0)
    say(f"# b3_verify_multiple_grouped vs the ungrouped call on the expanded inputs, one call in flight, median of {reps} after 2 warm-up rounds")
    say(f"# card: {card()}")
    rnd = random.Random(0x6A0)
    sks = [rnd.randrange(1, R) for _ in range(POOL)]
    pool = eng.g1_mul_gen(sks)
    tbl = mb.KeyTable(eng)
    _, st = tbl.append(pool.reshape(-1), compressed=False, validate=True)
    assert not st.any()
    shapes = [("512 x 1 key, 1 message", 512, 1, 1, False), ("8192 x 1 key, 64 messages", 8192, 1, 64, False),
              ("8192 x 128 table keys, 64 messages", 8192, 128, 64, True), ("8192 x 128 table keys, all distinct", 8192, 128, 8192, True)]
    say(f"{'shape':<38} | {'grouped host':>12} {'dev':>8} | {'expanded host':>13} {'dev':>8} | {'grouped / expanded':>18}")
    stage_rows = []
    for si, (label, n, nk, n_msgs, table) in enumerate(shapes):
        b = synth(eng, pool, sks, n, nk, n_msgs, 0x6A00 + si)
        kidx = b["idx"].reshape(-1)
        keys = kidx if table else np.ascontiguousarray(pool[kidx]).reshape(-1)
        t_ = tbl if table else None
        blob, moff, xblob, xoff = b"".join(b["msgs"]), offs(b["msgs"]), b"".join(b["ex"]), offs(b["ex"])

        def grouped():
            return eng.verify_multiple_grouped(t_, b["sigs"], keys, b["pk_off"], blob, moff, b["mi"], b["scalars"], want_gt=True)

        def expanded():
            if table:
                return eng.verify_multiple_indexed(tbl, b["sigs"], keys, b["pk_off"], xblob, xoff, b["scalars"], want_gt=True)
            return eng.verify_multiple(b["sigs"], keys, b["pk_off"], xblob, xoff, b["scalars"], want_gt=True)

        t = {"g": [], "g_dev": [], "x": [], "x_dev": []}
        for r in range(reps + 2):
            order = (("g", grouped), ("x", expanded)) if r % 2 == 0 else (("x", expanded), ("g", grouped))
            res = {}
            for k, fn in order:
                t0 = time.perf_counter()
                res[k] = fn()
                t1 = time.perf_counter()
                if r >= 2:
                    t[k].append((t1 - t0) * 1e3)
                    t[k + "_dev"].append(eng.last_kernel_ms(0))
            assert res["g"] == res["x"] and res["g"][0] and res["g"][1] == -1, label
        m = {k: float(np.median(v)) for k, v in t.items()}
        say(f"{label:<38} | {m['g']:>12.2f} {m['g_dev']:>8.2f} | {m['x']:>13.2f} {m['x_dev']:>8.2f} | {m['g'] / m['x']:>18.3f}")
        eng.set_serial(True)
        try:
            for k, fn in (("grouped", grouped), ("expanded", expanded)):
                fn()
                stage_rows.append((label, k, eng.stage_ms()))
        finally:
            eng.set_serial(False)
    say("# times in ms; 'grouped / expanded' = ratio of the host-clock medians")
    say("")
    say("# per-stage device ms, one serial call each (stages one after another on the context's stream)")
    names = list(stage_rows[0][2])
    say(f"{'shape':<38} {'call':<9} | " + " ".join(f"{s[:14]:>14}" for s in names))
    for label, k, st_ in stage_rows:
        say(f"{label:<38} {k:<9} | " + " ".join(f"{st_[s]:>14.3f}" for s in names))
    say("# stage names: " + ", ".join(names))
    if out_path:
        os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
        with open(out_path, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
