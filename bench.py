#!/usr/bin/env python3
"""bench.py -- verified signature-sets/s of verify_multiple_aggregate_signatures on B200.

Usage:  python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
  * workload at N = 1: BASELINE.json configs[3] -- 8192 attestation sets x 128 public keys, distinct random
    32-byte messages, 63-bit batch scalars (C4).  For N > 1 every rank keeps 8192 sets (weak scaling), so N = 8
    is BASELINE.json configs[4] (2^16 sets, NCCL combine of the 592-byte partial Miller products).
  * one call = one full verification of a C4 batch: G2 subgroup checks, G1 key aggregation, [c]apk, hash_to_G2,
    [c]sig sum, n+8 Miller loops, Fp12 product, (all-gather,) one final exponentiation, accept bit.
  * a step = one such call on EACH of --inflight (default 8) contexts per GPU, running concurrently.  Four are enough to
    saturate one B200 (profiles/r2_calls_in_flight.txt: 1.13 M sets/s with one call in flight, 1.40 M with two, 1.52 M with
    three, 1.60 M with four, 1.60-1.62 M with 6..16); eight give the sharded run the slack that hides the other ranks' jitter
    at the all-gather (N = 8: 12.08 M sets/s with eight, 11.57 M with four).  One b3_ctx + one
    host thread per call, the reference's own threading model (re-entrant types, callers parallelise externally).  A
    single 8192-set call is a chain of latency-bound kernels (~7 ms end to end) that cannot fill 148 SMs by itself;
    K steps = K x inflight full verifications of 8192 sets each.
  * keys: the reference pays PublicKey::from_bytes (decompression + key_validate, M/src/keys.rs:140-147) ONCE per validator
    and verification then works on decoded keys.  The drop-in equivalent is the device-resident KEY TABLE
    (b3_keytable_*: 2^20 validators = 100 MB of decoded keys in HBM, loaded once from 48-byte compressed keys, untimed);
    a set names its 128 keys by u32 index.  `byte_keys` reports the same metric with the 96-byte uncompressed keys passed
    to every call instead (round 1's headline path).
  * value  = sets verified per second, inputs resident in HBM (device-pointer C-ABI entry points).
             `one_batch_in_flight` reports the same metric with a single call at a time (call latency).
  * e2e    = same metric through the host-pointer C-ABI call (b3_verify_multiple_indexed; b3_sharded_begin/_finish at
             N > 1) with pinned HOST buffers: H2D of the step's inputs (signatures, key indices, offsets, messages, scalars)
             and D2H of accept + first_bad + GT inside the timed region.  `e2e.pageable` = the same from pageable host
             memory (what a Rust Vec<u8> is).
  * N > 1: every rank verifies its 8192-set shard; the 592-byte partials are combined by ONE ncclAllGather per step issued
    INSIDE the library (b3_comm_*, include/milagro_bls_b200.h); bench.py calls only C-ABI functions on the data path
    (torch.distributed is used for the barrier, the max-over-ranks of the timing and shipping the NCCL unique id).
  * roofline: bound = integer multiply pipe (IMAD); the peak is measured live with a pure IMAD.WIDE carry-chain
    probe (b3_imad_peak); HBM figures are reported next to it to show that memory is not binding.
  * cpu_baseline / --impl reference: the reference's CPU algorithm (oracle/ C restatement; the Rust crate cannot be
    built here -- no rustc) on all host cores, on a bounded sample of the same workload.
Only this file's cpu_baseline / --impl reference legs touch oracle/ -- never the measured GPU path.
"""
import argparse
import json
import os
# every context owns four CUDA streams; the default of 8 hardware work queues would alias the streams of concurrent
# batches onto shared queues (false dependencies between independent batches)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SETS_PER_GPU = 8192
KEYS_PER_SET = 128
POOL = 1 << 20            # validators in the key table (100 MB of decoded keys; Ethereum-mainnet order of magnitude)
MSG_LEN = 32
R_ORDER = 0x73eda753299d7d483339d80809a1d80553bda402fffe5bfeffffffff00000001
# algorithmic work per unit (SURVEY.md section 8d): 32x32->64 multiply-accumulates, 300 per Fp multiplication
MACS_PER_FP_MUL = 300
FP_MULS = {"g1_aggregate": 1400, "g2_parse_subgroup_check": 1170, "hash_to_g2_affine": 6700, "g1_scalar_mul_affine": 670 + 15,
           "g2_scalar_mul_sum": 1650, "miller_lines": 1800, "miller_accumulate": 3000, "miller_chain": 0, "final_exp": 0,
           "miller_lines_signature_sums": 0}
FP_MULS_PER_SET = 16400
# what this implementation actually executes per set (DESIGN.md section 4: inversion-free maps, bucket-method sum, split
# Miller loop), in the same unit -- reported beside the SURVEY figure so the fraction cannot flatter the kernels
EXEC_FP_MULS_PER_SET = 12900
# DRAM bytes (read + write) per launch at the C4 shape from the committed `ncu --set full` capture profiles/r2p_c4_full.txt
# (hash_to_G2: 0.26 MB of messages in, 2.36 MB of points out; the rest is write-back of its local-memory stack)
NCU_TRAFFIC_BYTES = {"hash_to_g2_affine": 532480 + 6281728, "miller_accumulate": 162431232 + 5712384, "g1_aggregate": 10587392 + 11520}
# 32x32->64 multiply-accumulates actually EXECUTED per unit (set / message / pair): IMAD.WIDE warp instructions x 32 lanes of the
# `ncu --set full --import-source on` capture of a 32768-set call, divided by its units (profiles/r2c_big32768_opcodes.txt).
# g1_aggregate is the byte-key kernel (parse + 2 Montgomery conversions + on-curve check per key on top of the 11-M mixed addition).
NCU_EXEC_MACS = {"hash_to_g2_affine": 1.255e6, "g2_parse_subgroup_check": 3.28e5, "g1_aggregate": 5.47e5, "g1_scalar_mul_affine": 1.87e5,
                 "miller_lines": 4.42e5, "miller_accumulate": 9.16e5}
CPU_PASSES = 4                # timed passes of the CPU baseline over its 2048-set sample (~10 s of CPU work per 4 cores)
B3_EXTRA_PAIRS = 8            # window sums of the bucket-method signature sum, each its own pair
BYTES_PER_SET = KEYS_PER_SET * 96 + 192 + MSG_LEN + 8          # algorithmic HBM bytes read per set


def splitmix64(seed):
    x = seed & (2**64 - 1)
    while True:
        x = (x + 0x9E3779B97F4A7C15) & (2**64 - 1)
        z = x
        z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & (2**64 - 1)
        z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & (2**64 - 1)
        yield z ^ (z >> 31)


def synth_pool(eng, seed):
    """The validator set: POOL secret keys and their public keys pk = [sk]G1 (GPU helper b3_g1_mul_gen; input synthesis, untimed)."""
    import numpy as np
    rs = np.random.RandomState(seed & 0x7fffffff)
    raw = rs.bytes(32 * POOL)
    sks = [1 + int.from_bytes(raw[32 * i:32 * i + 32], "big") % (R_ORDER - 1) for i in range(POOL)]
    pool = np.concatenate([eng.g1_mul_gen(sks[i:i + 65536]) for i in range(0, POOL, 65536)])      # (POOL, 96)
    return sks, pool


def synth_inputs(eng, sks, pool, n_sets, n_keys, seed, rank=0):
    """Synthetic, VALID signature sets (SURVEY.md section 8d): set j = n_keys distinct validators, sig_j = [sum sk]H(m_j)
    (GPU helper b3_g2_mul; input synthesis, not timed)."""
    import numpy as np
    rs = np.random.RandomState((seed + 7919 * rank) & 0x7fffffff)
    idx = rs.randint(0, POOL, size=(n_sets, n_keys)).astype(np.uint32)                         # (n_sets, n_keys), distinct within a set:
    while True:
        srt = np.sort(idx, axis=1)
        dup = np.nonzero((srt[:, 1:] == srt[:, :-1]).any(axis=1))[0]
        if len(dup) == 0:
            break
        idx[dup] = rs.randint(0, POOL, size=(len(dup), n_keys)).astype(np.uint32)
    msgs = rs.randint(0, 256, size=(n_sets, MSG_LEN), dtype=np.uint8)
    msgs[:, 0] = rank
    msgs[:, 1:5] = np.arange(n_sets, dtype=">u4").view(np.uint8).reshape(n_sets, 4)            # all distinct
    agg = [sum(sks[i] for i in row) % R_ORDER for row in idx.tolist()]
    H = eng.hash_to_g2([m.tobytes() for m in msgs])
    sigs = eng.g2_mul(H.reshape(-1), agg)                        # (n_sets, 192)
    pks = pool[idx.reshape(-1)]                                  # (n_sets*n_keys, 96)
    pk_off = np.arange(0, n_sets * n_keys + 1, n_keys, dtype=np.uint32)
    msg_off = np.arange(0, n_sets * MSG_LEN + 1, MSG_LEN, dtype=np.uint32)
    return {"sigs": np.ascontiguousarray(sigs.reshape(-1)), "pks": np.ascontiguousarray(pks.reshape(-1)), "pk_off": pk_off,
            "idx": np.ascontiguousarray(idx.reshape(-1)), "msgs": np.ascontiguousarray(msgs.reshape(-1)), "msg_off": msg_off, "n": n_sets}


def draw_scalars(n, seed):
    import numpy as np
    from milagro_bls_b200 import SeededRng, draw_scalar
    rng = SeededRng(seed)
    return np.array([draw_scalar(rng) for _ in range(n)], dtype=np.uint64)


class ClockSampler:
    """Samples the SM clock and the throttle reasons of one GPU during the timed region (B200_PROFILING.md recipe).  NVML is
    read in-process (nvidia_ml_py) every 20 ms: a polling `nvidia-smi -lms 100` process costs the GPU it watches ~3 % at
    N = 8 (every rank waits for the slowest at the all-gather); the CLI is the fallback when the module is missing."""

    REASONS = (("hw_slowdown", 0x8), ("hw_thermal_slowdown", 0x40), ("sw_thermal_slowdown", 0x20), ("sw_power_cap", 0x4))

    def __init__(self, index):
        self.index, self.sm, self.mx, self.reasons, self.proc, self.stop_ev, self.t = index, [], [], set(), None, threading.Event(), None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.nv = None
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read_cli, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        nv = self.nv
        while not self.stop_ev.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                self.mx.append(float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)))
                bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(nv, "nvmlDeviceGetCurrentClocksEventReasons")
                           else nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for name, bit in self.REASONS:
                    if bits & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self.stop_ev.wait(0.02)

    def _read_cli(self):
        for line in self.proc.stdout:
            r = [c.strip() for c in line.split(",")]
            try:
                self.sm.append(float(r[0])); self.mx.append(float(r[1]))
                for k, (name, _) in enumerate(self.REASONS):
                    if r[3 + k].lower().startswith("active"):
                        self.reasons.add(name)
            except Exception:
                pass

    def stop(self):
        self.stop_ev.set()
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.t:
            self.t.join(timeout=2)
        sm = sorted(self.sm)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(self.mx) if self.mx else None, "reasons": sorted(self.reasons),
                "samples": len(sm), "source": "nvml" if getattr(self, "nv", None) else "nvidia-smi"}


# ------------------------------------------------------------------------------------------------- CPU baseline
def cpu_reference_run(sample_sets, n_keys, seed, threads=None):
    """Times the CPU restatement of the reference's algorithm (oracle/) on `sample_sets` sets of the same shape,
    T independent single-threaded instances on disjoint chunks (the reference has no threads).  Returns a dict."""
    from oracle import cpu_baseline
    return cpu_baseline.run(sample_sets, n_keys, seed, threads)


def reference_main(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import numpy as np  # noqa: F401
    cores = os.cpu_count() or 1
    sample = max(cores, args.ref_sets)
    times, last = [], None
    for it in range(args.warmup + args.steps):
        last = cpu_reference_run(sample, KEYS_PER_SET, 0xB200, cores)
        if it >= args.warmup:
            times.append(last["seconds"])
    sec = sum(times) / max(len(times), 1)
    value = sample / sec
    line = {"impl": "reference", "metric": "verified sig-sets/s (verify_multiple_aggregate_signatures, 128 keys/set)", "value": value,
            "unit": "sets/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64 (6x64-bit Montgomery limbs, __int128)",
            "data": "synthetic",
            "config": {"workload": f"verify_multiple_aggregate_signatures: {SETS_PER_GPU} sets x {KEYS_PER_SET} keys per GPU (C4/C5)",
                       "sample_sets_per_step": sample, "keys_per_set": KEYS_PER_SET},
            "cpu_baseline": {"value": value, "unit": "sets/s", "cores": last["threads"], "kind": last["kind"],
                             "sample": f"{sample} sets x {KEYS_PER_SET} keys per step, {last['threads']} independent single-threaded instances"},
            "e2e": {"value": value, "unit": "sets/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--sets", type=int, default=SETS_PER_GPU, help="sets per GPU (default: the C4 shape)")
    ap.add_argument("--keys", type=int, default=KEYS_PER_SET)
    ap.add_argument("--ref-sets", type=int, default=2048,
                    help="sets per step of the CPU reference arm / cpu_baseline sample (~20 s of CPU work on 16 cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--inflight", type=int, default=8,
                    help="verification batches in flight per GPU (one b3_ctx + host thread each; 1 = one call at a time)")
    ap.add_argument("--pipeline-depth", type=int, default=1, choices=[1, 2],
                    help="N > 1: a lane finishes call k after beginning call k + depth (the all-gather of a step then has depth call times to complete)")
    ap.add_argument("--h2c-msgs", type=int, default=65536, help="messages per hash_to_G2 batch of the second metric")
    ap.add_argument("--no-next-rows", action="store_true", help="skip the SURVEY 8(f) rows (decompression, aggregation, per-item verification)")
    ap.add_argument("--breakdown", action="store_true", help="print the per-stage device times to stderr")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last headline step and the last hash_to_G2 batch returned as DIR/<name>.npy "
                         "(float32 / float64; fixed inputs, so two builds can be compared output for output)")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            raise SystemExit("bench.py: --dump-outputs dumps the GPU path; the reference arm has no outputs to dump")
        return reference_main(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import milagro_bls_b200 as mb

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product has no CPU path")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    comm = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
        # the library's own communicator (b3_comm_create): rank 0 makes the NCCL unique id, torch.distributed only ships it
        uid = torch.zeros(128, dtype=torch.uint8, device=dev)
        if rank == 0:
            uid.copy_(torch.from_numpy(np.frombuffer(mb.nccl_unique_id(), dtype=np.uint8).copy()))
        dist.broadcast(uid, 0)
        comm = mb.Comm(local_rank, world, rank, uid.cpu().numpy().tobytes(), lanes=max(1, args.inflight))
    eng = mb.Engine(local_rank)
    try:
        _bench(eng, comm, args, world, rank, local_rank, dev)    # every tensor made on the library's stream dies in here
    finally:
        torch.cuda.synchronize()
        torch.cuda.set_stream(torch.cuda.default_stream(dev))
        if comm is not None:
            comm.close()
        eng.close()                                              # ... before the stream itself is destroyed
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


class Lane:
    """One verification context (b3_ctx = its own CUDA streams and scratch) with its own synthetic batch.  The reference's
    types are re-entrant and its callers parallelise externally (SURVEY.md section 8b, threading): concurrent batches on
    separate contexts are the drop-in equivalent, and they are what keeps the GPU full while one batch is in its serial
    tail (closing Miller chain, final exponentiation).  Inputs are held three times: resident in HBM, in pinned host
    memory and in pageable host memory; keys both as u32 indices into the shared key table and as 96-byte records."""

    KEYS = ("sigs", "pks", "idx", "pk_off", "msgs", "msg_off")

    def __init__(self, local_rank, dev, table, sks, pool, n, nk, seed, rank, tag, index):
        import numpy as np
        import torch
        import milagro_bls_b200 as mb
        self.eng = mb.Engine(local_rank)
        self.index = index
        self.table = table
        self.stream = torch.cuda.ExternalStream(int(self.eng.L.b3_ctx_stream(self.eng.handle)), device=dev)
        inp = synth_inputs(self.eng, sks, pool, n, nk, seed, rank)
        scal = draw_scalars(n, b"bench-%d-%d" % (rank, tag))
        as_i32 = lambda a: a.view(np.int32) if a.dtype == np.uint32 else a          # torch has no uint32 arithmetic; bits are what matter
        with torch.cuda.stream(self.stream):
            self.d = {k: torch.from_numpy(as_i32(inp[k])).to(dev) for k in self.KEYS}
            self.d["scal"] = torch.from_numpy(scal.view(np.int64)).to(dev)
            self.stream.synchronize()
        self.pin = {k: torch.from_numpy(as_i32(inp[k])).pin_memory() for k in self.KEYS}
        self.pin["scal"] = torch.from_numpy(scal.view(np.int64)).pin_memory()
        self.page = {k: inp[k] for k in self.KEYS}                                   # plain numpy = pageable host memory
        self.page["scal"] = scal
        nb = lambda t: int(t.numel() * t.element_size())
        self.h2d_bytes = {"table": sum(nb(self.pin[k]) for k in ("sigs", "idx", "pk_off", "msgs", "msg_off", "scal")),
                          "bytes": sum(nb(self.pin[k]) for k in ("sigs", "pks", "pk_off", "msgs", "msg_off", "scal"))}

    def host(self, src):
        """numpy views of the host copy `src` in {"pinned", "pageable"} (uint32 / uint64 dtypes as the API wants them)."""
        import numpy as np
        if src == "pageable":
            return self.page
        h = {k: v.numpy() for k, v in self.pin.items()}
        for k in ("idx", "pk_off", "msg_off"):
            h[k] = h[k].view(np.uint32)
        h["scal"] = h["scal"].view(np.uint64)
        return h

    def partial_dev(self, n, base, d_partial, keys="bytes"):
        d = self.d
        if keys == "table":
            self.eng.verify_multiple_indexed_partial_dev(self.table, d["sigs"].data_ptr(), d["idx"].data_ptr(), d["pk_off"].data_ptr(),
                                                         d["msgs"].data_ptr(), d["msg_off"].data_ptr(), d["scal"].data_ptr(), n, base, d_partial)
        else:
            self.eng.verify_multiple_partial_dev(d["sigs"].data_ptr(), d["pks"].data_ptr(), d["pk_off"].data_ptr(), d["msgs"].data_ptr(),
                                                 d["msg_off"].data_ptr(), d["scal"].data_ptr(), n, base, d_partial)

    def close(self):
        self.d = self.pin = self.page = None
        self.eng.close()


def _bench(eng, comm, args, world, rank, local_rank, dev):
    import numpy as np
    import torch
    import milagro_bls_b200 as mb
    n, nk = args.sets, args.keys
    S = max(1, args.inflight)
    # every torch op of the benchmark (L2 flush, timing events) runs on the stream of `eng`
    lib_stream = torch.cuda.ExternalStream(int(eng.L.b3_ctx_stream(eng.handle)), device=dev)
    torch.cuda.set_stream(lib_stream)
    # the validator set and its device-resident key table: PublicKey::from_bytes (decompress + key_validate) ONCE per validator
    t0 = time.perf_counter()
    sks, pool = synth_pool(eng, 0xB200)
    c48 = np.concatenate([eng.g1_compress(pool[i:i + 65536].reshape(-1))[0].reshape(-1, 48) for i in range(0, POOL, 65536)])
    table = mb.KeyTable(eng, POOL)
    t1 = time.perf_counter()
    for i in range(0, POOL, 262144):
        first, st = table.append(c48[i:i + 262144].reshape(-1), compressed=True, validate=True)
        assert first == i and not st.any(), "every synthetic validator key must decompress and validate"
    table_s = time.perf_counter() - t1
    back, st = table.get(np.array([0, 1, POOL // 2, POOL - 1], dtype=np.uint32))
    assert not st.any() and back.tobytes() == pool[[0, 1, POOL // 2, POOL - 1]].tobytes(), "key table round trip"
    lanes = [Lane(local_rank, dev, table, sks, pool, n, nk, 0xB200 + 0x101 * t, rank, t, t) for t in range(S)]
    del sks, pool, c48
    setup = {"validators": POOL, "table_bytes": 96 * POOL, "table_load_s": table_s, "table_load_keys_per_s": POOL / table_s,
             "table_load": "b3_keytable_append from 48-byte compressed keys (decompression + key_validate), host pointers, wall clock; paid once",
             "synthesis_s": time.perf_counter() - t0}
    try:
        _bench_lanes(eng, comm, table, lanes, setup, args, world, rank, local_rank, dev)
    finally:
        torch.cuda.synchronize()
        for ln in lanes:
            ln.close()
        table.close()


def _bench_next_rows(eng, lane, dev, n, nk):
    """SURVEY.md 8(f): batched decompression + validation (PublicKey::from_bytes / Signature::from_bytes), signature aggregation,
    per-item verification.  Host-pointer calls are timed by wall clock around the synchronous C-ABI call (H2D/D2H inside);
    the per-item verification runs on the lane's device-resident C4 batch and is timed by the library's CUDA events.
    Each row carries a size-independent parity property checked here (round trip / all items accept); bit-exact parity with
    the oracle is in tests/test_gpu_parity.py."""
    import numpy as np
    import torch
    from milagro_bls_b200 import _lib
    peak = eng.imad_peak(wide=True)
    out = {}

    def wall(fn, reps=3):
        fn()
        t0 = time.perf_counter()
        for _ in range(reps):
            r = fn()
        return (time.perf_counter() - t0) / reps, r

    def row(name, units, secs, fp_muls, extra=None):
        d = {"value": units / secs, "unit": name.split(":")[1], "units_per_call": units, "ms_per_call": secs * 1e3,
             "algorithmic_fp_muls_per_unit": fp_muls, "imad_frac": units / secs * fp_muls * MACS_PER_FP_MUL / peak}
        d.update(extra or {})
        out[name.split(":")[0]] = d

    keys96 = lane.pin["pks"].numpy()[:96 * 65536]
    nkeys = len(keys96) // 96
    c48, st = eng.g1_compress(keys96)
    assert not st.any()
    secs, (back, st) = wall(lambda: eng.g1_decompress(c48, validate=True))
    assert not st.any() and back.tobytes() == keys96.tobytes(), "G1 compress -> decompress round trip"
    row("g1_decompress_validate:keys/s", nkeys, secs, 490 + 1000, {"timing": "wall clock, host pointers (48 B in, 96 B + status out per key)"})
    sig192 = lane.pin["sigs"].numpy()
    nsig = len(sig192) // 192
    c96, st = eng.g2_compress(sig192)
    assert not st.any()
    secs, (back, st) = wall(lambda: eng.g2_decompress(c96))
    assert not st.any() and back.tobytes() == sig192.tobytes(), "G2 compress -> decompress round trip"
    row("g2_decompress:signatures/s", nsig, secs, 1100, {"timing": "wall clock, host pointers (96 B in, 192 B + status out per signature)"})
    off = np.arange(0, nsig + 1, 4, dtype=np.uint32)
    secs, (agg, st) = wall(lambda: eng.g2_aggregate(sig192, off))
    assert not st.any()
    row("g2_aggregate:signatures/s", nsig, secs, 30, {"signatures_per_aggregate": 4, "timing": "wall clock, host pointers"})
    # per-item verification (fast_aggregate_verify of every set of the resident batch: nk keys per item, one final exponentiation each)
    d = lane.d
    acc = torch.zeros(n, dtype=torch.int32, device=dev)
    stt = torch.zeros(n, dtype=torch.int32, device=dev)
    torch.cuda.synchronize()
    best = None
    for _ in range(3):
        lane.eng.verify_batch_dev(_lib.ITEM_FAST_AGGREGATE, d["sigs"].data_ptr(), d["pks"].data_ptr(), d["pk_off"].data_ptr(),
                                  d["msgs"].data_ptr(), d["msg_off"].data_ptr(), n, acc.data_ptr(), stt.data_ptr())
        ms = lane.eng.last_kernel_ms(0)
        best = ms if best is None else min(best, ms)
    torch.cuda.synchronize()
    assert int(acc.sum()) == n and not bool(stt.any()), "every set of the valid batch verifies on its own"
    row("verify_batch_fast_aggregate:items/s", n, best * 1e-3, 1400 + 6700 + 1170 + 12260 + 8000,
        {"keys_per_item": nk, "timing": "CUDA events of the call, inputs resident in HBM; best of 3"})
    return out


def _bench_lanes(eng, comm, table, lanes, setup, args, world, rank, local_rank, dev):
    import numpy as np
    import torch
    import torch.distributed as dist
    import milagro_bls_b200 as mb
    n, nk = args.sets, args.keys
    S = len(lanes)
    PB = mb._lib.PARTIAL_BYTES
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    base = rank * n
    stage_acc, stage_lock = {}, threading.Lock()

    by_rank = []               # ms per step of every rank, one list per timed region (N > 1)
    call_events = []           # (start, end) CUDA events around every call of a one-batch-at-a-time run (after its L2 flush)

    def add_stages(e):
        st = e.stage_ms()
        with stage_lock:
            for k, v in st.items():
                stage_acc[k] = stage_acc.get(k, 0.0) + v

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def run_steps(steps, use_lanes, src="dev", keys="table", flush_l2=False, want_gt=False):
        """`steps` steps; a step = ONE full verification of a C4-shaped batch ON EVERY LANE (len(use_lanes) concurrent calls, each
        on its own context and host thread), batch i on lane i % L.  src: "dev" = inputs resident in HBM (device-pointer entries),
        "pinned" / "pageable" = host buffers through the host-pointer entries (H2D + D2H inside the call).  keys: "table" = u32
        indices into the device-resident key table, "bytes" = 96-byte uncompressed keys.
        N = 1: b3_verify_multiple[_indexed] (host pointers) or b3_verify_multiple[_indexed]_dev (device pointers).
        N > 1: b3_sharded_begin / b3_sharded_finish -- the all-gather of a step's partials is issued inside the library; a lane
        begins call k + 1 before it finishes call k, so the collective has a whole call time to complete."""
        L = len(use_lanes)
        B = steps * L
        partials = torch.zeros(max(B, 1), PB, dtype=torch.uint8, device=dev)
        torch.cuda.current_stream().synchronize()
        results = [None] * B
        errors = []
        call_events.clear()
        tbl = table if keys == "table" else None
        kname = "idx" if keys == "table" else "pks"

        def lane_main(t):
            ln = use_lanes[t]
            e = ln.eng
            pending = []
            try:
                with torch.cuda.stream(ln.stream):
                    h = ln.host(src) if src != "dev" else None
                    d = ln.d
                    for i in range(t, B, L):
                        if flush_l2:
                            flush.fill_(1)                          # evict L2 between iterations (single-lane mode only)
                            ln.stream.synchronize()
                            ca, cb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                            ca.record()                             # the call's own span, without the flush (ln.stream is current)
                            call_events.append((ca, cb))
                        if world > 1:
                            if src == "dev":
                                tk = e.sharded_begin_dev(comm, ln.index, tbl, d["sigs"].data_ptr(), d[kname].data_ptr(), d["pk_off"].data_ptr(),
                                                         d["msgs"].data_ptr(), d["msg_off"].data_ptr(), d["scal"].data_ptr(), n, base)
                            else:
                                tk = e.sharded_begin(comm, ln.index, tbl, h["sigs"], h[kname], h["pk_off"], h["msgs"], h["msg_off"], h["scal"], base)
                            add_stages(e)
                            pending.append((i, tk))
                            if L == 1 and flush_l2:                  # one call at a time: no pipelining
                                results[i] = e.sharded_finish(comm, ln.index, tk, want_gt=want_gt)
                                add_stages(e)
                                pending.clear()
                                call_events[-1][1].record()
                            while len(pending) > args.pipeline_depth:   # finish call k only after beginning call k + depth
                                j, tj = pending.pop(0)
                                results[j] = e.sharded_finish(comm, ln.index, tj, want_gt=want_gt)
                                add_stages(e)
                            continue
                        if src != "dev":                              # the reference-facing call on host pointers
                            if keys == "table":
                                results[i] = e.verify_multiple_indexed(ln.table, h["sigs"], h["idx"], h["pk_off"], h["msgs"], h["msg_off"], h["scal"],
                                                                       want_gt=True)
                            else:
                                results[i] = e.verify_multiple(h["sigs"], h["pks"], h["pk_off"], h["msgs"], h["msg_off"], h["scal"], want_gt=True)
                            add_stages(e)
                            if flush_l2:
                                call_events[-1][1].record()
                            continue
                        results[i] = e.verify_multiple_dev(tbl, d["sigs"].data_ptr(), d[kname].data_ptr(), d["pk_off"].data_ptr(), d["msgs"].data_ptr(),
                                                           d["msg_off"].data_ptr(), d["scal"].data_ptr(), n, want_gt=True)
                        add_stages(e)
                        if flush_l2:
                            call_events[-1][1].record()
                    for j, tj in pending:
                        results[j] = e.sharded_finish(comm, ln.index, tj, want_gt=want_gt)
                        add_stages(e)
            except BaseException as ex:                              # noqa: BLE001
                errors.append(ex)

        threads = [threading.Thread(target=lane_main, args=(t,), daemon=True) for t in range(L)]
        for th in threads:
            th.start()
        for th in threads:
            th.join()
        if errors:
            raise errors[0]
        return results

    def total_launches():
        return eng.launches + sum(ln.eng.launches for ln in lanes)

    def timed(steps, warmup, use_lanes, **kw):
        if world > 1 and len(use_lanes) != S:
            raise RuntimeError("at N > 1 every step must use all lanes of the communicator")
        for r in run_steps(warmup, use_lanes, **kw):
            assert r[0] and r[1] == -1, "verification of the valid synthetic batch must accept"
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        launches0 = total_launches()
        with stage_lock:
            stage_acc.clear()
        e0.record()                                   # device idle (barrier above): the timestamp is "now"
        res = run_steps(steps, use_lanes, **kw)
        torch.cuda.synchronize()                      # every lane's streams
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if kw.get("flush_l2") and len(call_events) == steps * len(use_lanes):
            ms = sum(a.elapsed_time(b) for a, b in call_events)          # the calls themselves; the 256 MiB flushes between them excluded
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            allt = [torch.zeros_like(t) for _ in range(world)]
            dist.all_gather(allt, t)
            by_rank.append([round(float(x.item()) / steps, 3) for x in allt])
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        for r in res:
            assert r[0] and r[1] == -1, "verification of the valid synthetic batch must accept"
        with stage_lock:
            st = {k: v / (steps * len(use_lanes)) for k, v in stage_acc.items()}
        return float(t.item()), total_launches() - launches0, st, res[-len(use_lanes):]      # results of the last step

    W = max(args.warmup, 3)
    K = args.steps
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    # headline: S batches in flight, inputs resident in HBM, keys named by index into the resident key table
    ms_res, launches, stages_pipe, last = timed(K, W, lanes)
    clocks = sampler.stop() if rank == 0 else None
    if os.environ.get("B3_BENCH_DIAG"):                 # diagnostic: the headline region again, now without the clock sampler
        m2 = timed(K, W, lanes)[0]
        m3 = timed(K, W, lanes)[0]
        if rank == 0 and os.environ.get("B3_BENCH_PRINT_HEADLINE"):
            print("headline_region ms_per_step", [round(x / K, 3) for x in (ms_res, m2, m3)], "sets/s",
                  [round(n * world * S * K / (x * 1e-3)) for x in (ms_res, m2, m3)], flush=True)
        if rank == 0:
            print(json.dumps({"diag_ms_per_step_by_rank": by_rank}), flush=True)
        return
    colls0 = comm.collectives if comm is not None else 0
    # e2e: the same from pinned HOST buffers through the host-pointer C ABI (H2D + D2H inside the timed region) ...
    ms_e2e, _, _, _ = timed(K, W, lanes, src="pinned")
    colls = (comm.collectives - colls0) if comm is not None else 0
    # ... and from pageable host memory (what a Rust Vec<u8> is)
    ms_e2e_page, _, _, _ = timed(K, W, lanes, src="pageable")
    # the same two with the 96-byte uncompressed keys passed to every call (round 1's headline path)
    ms_res_b, _, _, _ = timed(K, W, lanes, keys="bytes")
    ms_e2e_b, _, _, _ = timed(K, W, lanes, src="pinned", keys="bytes")
    ms_e2e_b_page, _, _, _ = timed(K, W, lanes, src="pageable", keys="bytes")
    one = None
    stages = stages_serial = {}
    if world == 1:
        # one batch in flight (call latency), L2 flushed before every step: per-kernel spans for the roofline
        ms_one, _, stages, _ = timed(K, W, lanes[:1], flush_l2=True)
        ms_one_e2e, _, _, _ = timed(K, W, lanes[:1], src="pinned", flush_l2=True)
        ms_one_b, _, _, _ = timed(K, W, lanes[:1], keys="bytes", flush_l2=True)
        one = {"value": n * K / (ms_one * 1e-3), "ms_per_step": ms_one / K, "e2e_value": n * K / (ms_one_e2e * 1e-3),
               "e2e_ms_per_step": ms_one_e2e / K, "byte_keys_value": n * K / (ms_one_b * 1e-3), "byte_keys_ms_per_step": ms_one_b / K,
               "cache": "L2 flushed (256 MiB write) before every call; time = sum of the CUDA-event spans of the calls (flushes excluded)"}
        # untimed diagnostic pass: the same step with the independent stages serialised, for a clean per-stage breakdown
        lanes[0].eng.set_serial(True)
        with stage_lock:
            stage_acc.clear()
        run_steps(2, lanes[:1], flush_l2=True)
        with stage_lock:
            stages_serial = {k: v / 2 for k, v in stage_acc.items()}
        lanes[0].eng.set_serial(False)
    # correctness inside the bench (every run, every N): (1) the GT bytes of the valid batch are the same on every rank and for
    # both key forms; (2) a batch with one flipped message bit on the LAST rank rejects on every rank, with one GT everywhere;
    # (3) a non-subgroup signature on the last rank comes back as the GLOBAL first_bad on every rank
    ln = lanes[0]

    def one_call(keys="table"):
        if world > 1:
            # every lane of the communicator must take part in a step: lanes 1.. repeat their own valid batch
            return run_steps(1, lanes, keys=keys, want_gt=True)[0]
        return run_steps(1, lanes[:1], keys=keys, want_gt=True)[0]

    def same_everywhere(gt, what):
        if world == 1:
            return
        g = torch.from_numpy(np.frombuffer(gt, dtype=np.uint8).copy()).to(dev)
        allg = [torch.empty_like(g) for _ in range(world)]
        dist.all_gather(allg, g)
        assert all(bool((x == allg[0]).all()) for x in allg), f"{what}: GT differs between ranks"

    ok_v, fb_v, gt_v = one_call("table")
    ok_b, fb_b, gt_b = one_call("bytes")
    assert ok_v and ok_b and fb_v == -1 and gt_v == gt_b, "key-table and byte-key calls must give the same GT"
    same_everywhere(gt_v, "valid batch")
    tamper = rank == world - 1
    keep_m, keep_s = ln.d["msgs"], ln.d["sigs"]
    if tamper:
        bad = keep_m.clone()
        bad[5] ^= 1
        torch.cuda.synchronize()
        ln.d["msgs"] = bad
    ok_t, fb_t, gt_t = one_call("table")
    ln.d["msgs"] = keep_m
    assert not ok_t and fb_t == -1 and gt_t != gt_v, "tampered batch must reject (on every rank)"
    same_everywhere(gt_t, "tampered batch")
    # (3) an on-curve point outside G2 as signature 7 of the last rank: b3_g2_decompress of random x coordinates yields curve
    # points, which lie in the order-r subgroup with probability ~2^-381
    if tamper:
        rs = np.random.RandomState(77)
        rogue = None
        for _ in range(256):
            c = bytearray(rs.bytes(96))
            c[0] = 0x80 | (c[0] & 0x0f)
            c[48] &= 0x0f
            pt, st = eng.g2_decompress(bytes(c))
            if st[0] == 0:
                rogue = pt.reshape(-1)
                break
        assert rogue is not None, "no on-curve point found"
        st, okg = eng.g2_subgroup_check(rogue)
        assert st[0] == 0 and not okg[0], "random curve point must fail the G2 subgroup check"
        bad_s = keep_s.clone()
        bad_s[7 * 192:8 * 192] = torch.from_numpy(rogue.copy()).to(dev)
        torch.cuda.synchronize()
        ln.d["sigs"] = bad_s
    ok_r, fb_r, _ = one_call("table")
    assert not ok_r and fb_r == (world - 1) * n + 7, f"non-subgroup signature: global first_bad expected {(world - 1) * n + 7}, got {fb_r}"
    ln.d["sigs"] = keep_s

    # second headline metric: hash_to_G2/s (b3_hash_to_g2_dev: SHA-256 xmd, SSWU, 3-isogeny, cofactor clearing, affine
    # normalisation and 192-byte wire output), 32-byte messages resident in HBM
    nh = args.h2c_msgs
    hmsgs = np.random.RandomState(5 + rank).randint(0, 256, size=nh * MSG_LEN, dtype=np.uint8)
    hm = torch.from_numpy(hmsgs).to(dev)
    ho = torch.arange(0, nh * MSG_LEN + 1, MSG_LEN, dtype=torch.int32, device=dev)
    hout = torch.empty(nh * 192, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    for _ in range(2):
        eng.hash_to_g2_dev(hm.data_ptr(), ho.data_ptr(), nh, hout.data_ptr())
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(K):
        eng.hash_to_g2_dev(hm.data_ptr(), ho.data_ptr(), nh, hout.data_ptr())
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_h2c = float(t.item())
    h2c_rate = nh * world * K / (ms_h2c * 1e-3)
    # the same through the host-pointer call (messages H2D, 192-byte points D2H inside)
    moff_h = np.arange(0, nh * MSG_LEN + 1, MSG_LEN, dtype=np.uint32)
    eng.hash_to_g2_blob(hmsgs, moff_h)
    t0 = time.perf_counter()
    for _ in range(K):
        hpts = eng.hash_to_g2_blob(hmsgs, moff_h)
    h2c_e2e_rate = nh * K / (time.perf_counter() - t0)
    assert hpts.tobytes() == hout.cpu().numpy().tobytes(), "host-pointer and device-pointer hash_to_G2 agree"

    # rows SURVEY.md 8(f) marks "next" (the callers / data formats either side of the path), measured on rank 0 at N = 1
    next_rows = _bench_next_rows(eng, lanes[0], dev, n, nk) if (world == 1 and not args.no_next_rows) else None

    total_sets = n * world                               # per call across the ranks
    rate = lambda ms: total_sets * S * K / (ms * 1e-3)
    value, e2e = rate(ms_res), rate(ms_e2e)
    h2d_bytes = lanes[0].h2d_bytes

    if rank != 0:
        return
    peak_mac = eng.imad_peak(wide=True)            # 32x32->64 MACs (IMAD.WIDE pairs) per second, measured live
    peak_imad = eng.imad_peak(wide=False)
    step_ms = ms_res / (K * S)                     # device time per 8192-set call in the headline region
    whole = FP_MULS_PER_SET * MACS_PER_FP_MUL * n / (step_ms * 1e-3)
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        hbm_peak, hbm_src = peaks["hbm_gbs"], "MEASURED_PEAKS.json"
    except Exception:
        hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
    hbm_achieved = BYTES_PER_SET * n / (step_ms * 1e-3) / 1e9
    roofline = {"bound": "imad", "unit": "GMAC/s (32x32->64 multiply-accumulate)", "peak": peak_mac / 1e9,
                "peak_source": "live probe b3_imad_peak(wide=1): IMAD.WIDE carry chains, all SMs",
                "plain_imad_peak_gops": peak_imad / 1e9, "macs_per_fp_mul": MACS_PER_FP_MUL,
                "whole_step": {"achieved": whole / 1e9, "frac": whole / peak_mac, "fp_muls_per_set": FP_MULS_PER_SET,
                               "frac_of_executed_work": whole / peak_mac * EXEC_FP_MULS_PER_SET / FP_MULS_PER_SET,
                               "executed_fp_muls_per_set_estimate": EXEC_FP_MULS_PER_SET},
                "hbm": {"achieved_gbs": hbm_achieved, "peak_gbs": hbm_peak, "frac": hbm_achieved / hbm_peak, "peak_source": hbm_src,
                        "algorithmic_bytes_per_set": BYTES_PER_SET},
                "stage_ms_pipelined": stages_pipe}
    if world == 1:
        # dominant kernel = the stage with the largest device time when run alone (serialised pass); its duration for the
        # roofline is the CUDA-event span inside the ONE-BATCH-IN-FLIGHT timed region (where it still shares the GPU with
        # the overlapped stages of its own batch, but not with a second batch -- spans of co-running batches are not
        # attributable to one kernel)
        dom = max((k for k in stages_serial if k in FP_MULS and FP_MULS[k] > 0), key=lambda k: stages_serial[k])
        dom_ms = stages[dom]
        units = n + (B3_EXTRA_PAIRS if dom.startswith("miller") else 0)
        achieved = FP_MULS[dom] * MACS_PER_FP_MUL * units / (dom_ms * 1e-3)
        per_stage = {k: {"ms_timed_region": stages[k], "ms_alone": stages_serial.get(k),
                         "ms_timed_region_pipelined": stages_pipe.get(k),
                         "frac_timed_region": FP_MULS[k] * MACS_PER_FP_MUL * n / (stages[k] * 1e-3) / peak_mac,
                         "frac_alone": FP_MULS[k] * MACS_PER_FP_MUL * n / (stages_serial[k] * 1e-3) / peak_mac if stages_serial.get(k) else None,
                         "executed_macs_per_unit_ncu": NCU_EXEC_MACS.get(k),
                         "frac_alone_executed": (NCU_EXEC_MACS[k] * n / (stages_serial[k] * 1e-3) / peak_mac
                                                 if (NCU_EXEC_MACS.get(k) and stages_serial.get(k)) else None)}
                     for k in stages if FP_MULS.get(k, 0) > 0 and stages[k] > 0}
        miller_ms = sum(stages_serial.get(k, 0.0) for k in ("miller_lines", "miller_accumulate", "miller_chain"))
        roofline.update({"kernel": dom, "achieved": achieved / 1e9, "frac": achieved / peak_mac,
                         "traffic": NCU_TRAFFIC_BYTES.get(dom) if (n == SETS_PER_GPU and nk == KEYS_PER_SET) else None,
                         "traffic_note": "DRAM bytes read + written per launch, ncu --set full capture under profiles/; the kernel is "
                                         "bound by the integer multiply pipe, not HBM",
                         "kernel_ms": dom_ms, "algorithmic_fp_muls_per_unit": FP_MULS[dom], "units_per_launch": units,
                         "frac_alone": per_stage[dom]["frac_alone"], "per_stage": per_stage,
                         "miller_loop_alone": {"ms": miller_ms, "fp_muls_per_pair": 4800,
                                               "what": "point chains of the n message pairs + accumulation of all n + 8 pairs + closing chain, each alone (serialised "
                                                       "pass); the point chains of the 8 signature-sum pairs (miller_lines_signature_sums, a latency-bound launch of "
                                                       "8 lane quads on its own stream) are listed apart",
                                               "frac": 4800 * MACS_PER_FP_MUL * (n + B3_EXTRA_PAIRS) / (miller_ms * 1e-3) / peak_mac if miller_ms else None},
                         "stage_ms": stages, "stage_ms_serialised": stages_serial,
                         "note": "kernel spans (stage_ms, frac) come from the one-batch-in-flight timed region (L2 flushed before every step): "
                                 "CUDA-event spans on the stream each stage runs on; independent stages of a batch overlap on separate streams, "
                                 "so they do not add up to the step.  stage_ms_serialised: same step with the stages run one after another "
                                 "(untimed pass).  stage_ms_pipelined: spans inside the headline region, where batches share the GPU.  "
                                 "whole_step is the headline region."})
        roofline["whole_step"]["frac_one_batch_in_flight"] = FP_MULS_PER_SET * MACS_PER_FP_MUL * n / (one["ms_per_step"] * 1e-3) / peak_mac
    else:
        roofline.update({"kernel": "whole step (per-kernel spans are measured at N = 1)", "achieved": whole / 1e9 / world,
                         "frac": whole / peak_mac / world, "traffic": None})
    cpu = cpu_h2c = None
    if not args.no_cpu_baseline and world == 1:
        ncpu = os.cpu_count() or 1
        try:
            cpu_reference_run(max(ncpu, args.ref_sets), nk, 0xB200, ncpu)      # warm-up pass
            passes = [cpu_reference_run(max(ncpu, args.ref_sets), nk, 0xB200, ncpu) for _ in range(CPU_PASSES)]
            c = passes[-1]
            c_sets, c_sec = sum(x["sets"] for x in passes), sum(x["seconds"] for x in passes)
            cpu = {"value": c_sets / c_sec, "unit": "sets/s", "cores": c["threads"], "kind": c["kind"],
                   "sample": f"{CPU_PASSES} passes over {c['sets']} sets x {nk} keys, {c['threads']} independent single-threaded instances, "
                             f"{c_sec:.1f} s wall = {c_sec * c['threads']:.0f} core-seconds"}
        except Exception as ex:                                        # noqa: BLE001
            cpu = {"value": None, "unit": "sets/s", "cores": 0, "kind": "port", "sample": f"unavailable: {ex}"}
        try:
            from oracle import cpu_baseline
            h = cpu_baseline.run_hash_to_g2(512 * ncpu, ncpu)
            cpu_h2c = {"value": h["msgs"] / h["seconds"], "unit": "hash_to_G2/s", "cores": h["threads"], "kind": h["kind"],
                       "sample": f"{h['msgs']} 32-byte messages, {h['threads']} independent single-threaded instances, {h['seconds']:.1f} s wall"}
        except Exception as ex:                                        # noqa: BLE001
            cpu_h2c = {"value": None, "unit": "hash_to_G2/s", "cores": 0, "kind": "port", "sample": f"unavailable: {ex}"}
    hb = h2d_bytes["table"]
    cache = (f"{S} batches in flight on {S} contexts, each with its own inputs and 160 MB of Miller-line scratch written and re-read per "
             f"step; keys gathered from a {96 * POOL / 1e6:.0f} MB table of {POOL} validators; no explicit flush" if S > 1 else
             "L2 flushed (256 MiB write) before every step")
    out = {"metric": "verified sig-sets/s (verify_multiple_aggregate_signatures, 128 keys/set)", "value": value, "unit": "sets/s",
           "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_res / K,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32 (12x32-bit Montgomery limbs, IMAD.WIDE)",
           "data": "synthetic",
           "config": {"workload": f"verify_multiple_aggregate_signatures: calls of {n} sets x {nk} keys per GPU "
                                  f"({'C4' if world == 1 else 'C5-style'}: {total_sets} sets per call over {world} GPU(s)), 32-byte distinct "
                                  f"messages, 63-bit scalars; keys = u32 indices into a device-resident table of {POOL} validator keys "
                                  f"(decoded once, as the reference's PublicKey::from_bytes); a step = {S} such calls in flight per GPU on {S} contexts",
                      "sets_per_call_per_gpu": n, "keys_per_set": nk, "sets_per_call": total_sets, "calls_per_step": S,
                      "sets_per_step": total_sets * S, "parallelism": f"set-sharded x{world}",
                      "collective": (f"one ncclAllGather of {S} x 592 B per rank per step, issued inside the library (b3_comm); "
                                     f"{colls} collectives in the e2e region of {K + W} steps") if world > 1 else None,
                      "batches_in_flight": S, "cache": cache, "key_table": setup},
           "e2e": {"value": e2e, "unit": "sets/s", "h2d_bytes_per_step": hb * world * S, "d2h_bytes_per_step": (576 + 16 + 8 * n + 36) * world * S,
                   "ms_per_step": ms_e2e / K, "host_memory": "pinned", "h2d_bytes_per_set": hb / n,
                   "pageable": {"value": rate(ms_e2e_page), "ms_per_step": ms_e2e_page / K}},
           "byte_keys": {"value": rate(ms_res_b), "ms_per_step": ms_res_b / K,
                         "e2e": {"value": rate(ms_e2e_b), "ms_per_step": ms_e2e_b / K, "h2d_bytes_per_step": h2d_bytes["bytes"] * world * S,
                                 "pageable": {"value": rate(ms_e2e_b_page), "ms_per_step": ms_e2e_b_page / K}},
                         "note": "the same calls with the 96-byte uncompressed keys passed (and parsed, converted, curve-checked) every time"},
           "one_batch_in_flight": one,
           "hash_to_g2": {"value": h2c_rate, "unit": "hash_to_G2/s", "messages_per_gpu": nh, "message_bytes": MSG_LEN,
                          "ms_per_batch": ms_h2c / K, "e2e_value": h2c_e2e_rate,
                          "e2e_note": "host-pointer b3_hash_to_g2 on rank 0: messages H2D and 192-byte points D2H inside, wall clock",
                          "imad_frac": h2c_rate / world * FP_MULS["hash_to_g2_affine"] * MACS_PER_FP_MUL / peak_mac,
                          "cpu_baseline": cpu_h2c},
           "next_rows": next_rows,
           "gpu_launches": launches, "clocks": clocks, "roofline": roofline, "cpu_baseline": cpu,
           "accept": bool(last[-1][0]),
           "ms_per_step_by_rank": by_rank if world > 1 else None,
           "checks": "valid batch: same GT on every rank and for both key forms; tampered message on the last rank: reject on every rank with one GT; non-subgroup signature on the last rank: global first_bad on every rank"}
    if args.breakdown:
        print(json.dumps({"overlapped": stages, "serialised": stages_serial, "pipelined": stages_pipe}, indent=1), file=sys.stderr)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last, hout.cpu().numpy().reshape(nh, 192))
    print(json.dumps(out), flush=True)


def dump_outputs(out_dir, last_step, h2c_points):
    """What a caller of the timed paths received, as float arrays (bytes 0..255 and small integers are exact):
    verify_*: one row per call of the last headline step (accept, first_bad and, at N = 1, the 576 GT bytes);
    hash_to_g2: the 192-byte wire points of every (n // 4096)-th of the n messages of the last batch, at most 4096 of them."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"verify_accept": np.array([r[0] for r in last_step], dtype=np.float32),
              "verify_first_bad": np.array([r[1] for r in last_step], dtype=np.float64),
              "hash_to_g2": h2c_points[::max(1, len(h2c_points) // 4096)][:4096].astype(np.float32)}
    if len(last_step[0]) == 3:
        arrays["verify_gt"] = np.stack([np.frombuffer(r[2], dtype=np.uint8) for r in last_step]).astype(np.float32)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


if __name__ == "__main__":
    sys.exit(main())
