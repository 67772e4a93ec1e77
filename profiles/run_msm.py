"""Device time of the signature-sum stage of verify_multiple (S = sum_j [c_j] sig_j: `g2_scalar_mul_sum`) across batch
sizes and scalar distributions, the stages serialised (b3_ctx_set_serial) so that the stage runs alone on the GPU.

Per (n, distribution): valid single-key sets synthesised on the GPU, one warm-up call, then the median of `reps` calls of the
library's own span of the stage (CUDA events).  Every call must accept.  Distributions: random 64-bit scalars, the
reference's draw (< 2^63), every set in one bucket of each window, and zero digits.  The card's name and power limit are
read in the same run.

usage: python profiles/run_msm.py [out.txt] [reps]"""
import os
import random
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import milagro_bls_b200 as mb  # noqa: E402

R = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name(0)}; nvidia-smi: {q}"


def scalars(kind, n, rnd):
    if kind == "random":
        return np.array([rnd.getrandbits(64) | 1 for _ in range(n)], dtype=np.uint64)
    if kind == "draw":
        return np.array([rnd.randrange(1, 1 << 63) for _ in range(n)], dtype=np.uint64)
    if kind == "one_bucket":
        return np.full(n, 0x9e3779b97f4a7c15, dtype=np.uint64)
    vals = [1, 1 << 56, 0x0100, 0x0100000000000001]
    return np.array([vals[j % 4] for j in range(n)], dtype=np.uint64)


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 7
    eng = mb.Engine(0)
    lines = [f"card: {card()}", f"g2_scalar_mul_sum, stages serialised, median of {reps} calls (ms)",
             f"{'sets':>6} " + " ".join(f"{k:>11}" for k in ("random", "draw", "one_bucket", "zero_digits"))]
    for n in (512, 2048, 8192, 32768):
        rnd = random.Random(n)
        sks = [rnd.randrange(1, R) for _ in range(n)]
        pk = eng.g1_mul_gen(sks).reshape(-1)
        msgs = [rnd.getrandbits(256).to_bytes(32, "big") for _ in range(n)]
        sig = eng.g2_mul(eng.hash_to_g2(msgs).reshape(-1), sks).reshape(-1)
        blob, moff = b"".join(msgs), list(range(0, 32 * n + 1, 32))
        row = []
        eng.set_serial(True)
        for kind in ("random", "draw", "one_bucket", "zero_digits"):
            sc = scalars(kind, n, rnd)
            t = []
            for _ in range(reps + 1):
                ok, _ = eng.verify_multiple(sig, pk, None, blob, moff, sc)
                assert ok, (n, kind)
                t.append(eng.stage_ms()["g2_scalar_mul_sum"])
            row.append(float(np.median(t[1:])))
        eng.set_serial(False)
        lines.append(f"{n:>6} " + " ".join(f"{v:>11.3f}" for v in row))
        print(lines[-1], flush=True)
    text = "\n".join(lines) + "\n"
    if out:
        os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
        with open(out, "w") as f:
            f.write(text)
    print(text)


if __name__ == "__main__":
    main()
