"""ctypes binding of the C ABI declared in include/milagro_bls_b200.h.

The product has NO CPU path: if the CUDA library is missing, or no sm_100 device is visible, every entry point
raises.  (The oracle under oracle/ is test infrastructure and is never imported from this package.)
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmilagro_bls_b200.so")

# error codes (include/milagro_bls_b200.h); -1..-8 mirror AmclError (A/errors.rs:1-11)
OK = 0
ERR_NAMES = {
    -1: "AggregateEmptyPoints", -2: "HashToFieldError", -3: "InvalidSecretKeySize", -4: "InvalidSecretKeyRange",
    -5: "InvalidPoint", -6: "InvalidG1Size", -7: "InvalidG2Size", -8: "InvalidYFlag", -100: "CudaError", -101: "BadArgument",
}
PARTIAL_BYTES = 592
ITEM_VERIFY, ITEM_FAST_AGGREGATE, ITEM_PRE_AGGREGATED = 0, 1, 2


class B3LibraryMissing(RuntimeError):
    pass


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise B3LibraryMissing(
            f"{LIB_PATH} not built: run `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc, sm_100a). There is no CPU fallback.")
    L = ctypes.CDLL(LIB_PATH)
    vp, sz, i32p, u8p = ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_int32), ctypes.c_void_p
    ip, i64p = ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int64)
    sigs = {
        "b3_ctx_create": ([ctypes.c_int, ctypes.POINTER(vp)], ctypes.c_int),
        "b3_ctx_destroy": ([vp], None),
        "b3_last_error": ([vp], ctypes.c_char_p),
        "b3_ctx_stream": ([vp], vp),
        "b3_ctx_launch_count": ([vp], ctypes.c_uint64),
        "b3_ctx_last_kernel_ms": ([vp, ctypes.c_int], ctypes.c_float),
        "b3_ctx_stage_ms": ([vp, ctypes.c_int], ctypes.c_float),
        "b3_stage_name": ([ctypes.c_int], ctypes.c_char_p),
        "b3_stage_count": ([], ctypes.c_int),
        "b3_ctx_set_serial": ([vp, ctypes.c_int], None),
        "b3_ctx_set_item_kernel": ([vp, ctypes.c_int], None),
        "b3_ctx_set_trusted_points": ([vp, ctypes.c_int], None),
        "b3_ctx_set_latency_mode": ([vp, ctypes.c_int], None),
        "b3_g1_decompress": ([vp, u8p, sz, ctypes.c_int, u8p, i32p], ctypes.c_int),
        "b3_g2_decompress": ([vp, u8p, sz, u8p, i32p], ctypes.c_int),
        "b3_g1_compress": ([vp, u8p, sz, u8p, i32p], ctypes.c_int),
        "b3_g2_compress": ([vp, u8p, sz, u8p, i32p], ctypes.c_int),
        "b3_g1_validate": ([vp, u8p, sz, i32p, i32p], ctypes.c_int),
        "b3_g2_subgroup_check": ([vp, u8p, sz, i32p, i32p], ctypes.c_int),
        "b3_g1_aggregate": ([vp, u8p, vp, sz, u8p, i32p], ctypes.c_int),
        "b3_g2_aggregate": ([vp, u8p, vp, sz, u8p, i32p], ctypes.c_int),
        "b3_hash_to_g2": ([vp, u8p, vp, sz, u8p, sz, u8p], ctypes.c_int),
        "b3_verify": ([vp, u8p, u8p, u8p, sz, ip, u8p], ctypes.c_int),
        "b3_fast_aggregate_verify": ([vp, u8p, u8p, sz, u8p, sz, ip, u8p], ctypes.c_int),
        "b3_fast_aggregate_verify_pre_aggregated": ([vp, u8p, u8p, u8p, sz, ip, u8p], ctypes.c_int),
        "b3_aggregate_verify": ([vp, u8p, u8p, u8p, vp, sz, ip, u8p], ctypes.c_int),
        "b3_verify_multiple": ([vp, u8p, u8p, vp, u8p, vp, vp, sz, ip, i64p, u8p], ctypes.c_int),
        "b3_verify_multiple_dev": ([vp, vp, vp, vp, vp, vp, vp, sz, ip, i64p, u8p], ctypes.c_int),
        "b3_verify_multiple_indexed_dev": ([vp, vp, vp, vp, vp, vp, vp, vp, sz, ip, i64p, u8p], ctypes.c_int),
        "b3_verify_multiple_locate": ([vp, sz, i32p, ctypes.POINTER(sz)], ctypes.c_int),
        "b3_verify_multiple_grouped": ([vp, vp, vp, vp, vp, vp, vp, sz, vp, vp, sz, ctypes.c_int, ip, i64p, u8p], ctypes.c_int),
        "b3_sig_precheck": ([vp, u8p, sz, i64p], ctypes.c_int),
        "b3_verify_multiple_checked": ([vp, u8p, vp, u8p, vp, vp, sz, ip, u8p], ctypes.c_int),
        "b3_keytable_create": ([vp, sz, ctypes.POINTER(vp)], ctypes.c_int),
        "b3_keytable_destroy": ([vp], None),
        "b3_keytable_size": ([vp], sz),
        "b3_keytable_append": ([vp, vp, u8p, sz, ctypes.c_int, ctypes.c_int, i32p, ctypes.POINTER(sz)], ctypes.c_int),
        "b3_keytable_get": ([vp, vp, vp, sz, u8p, i32p], ctypes.c_int),
        "b3_g1_aggregate_indexed": ([vp, vp, vp, vp, sz, u8p, i32p], ctypes.c_int),
        "b3_verify_multiple_indexed": ([vp, vp, u8p, vp, vp, u8p, vp, vp, sz, ip, i64p, u8p], ctypes.c_int),
        "b3_verify_multiple_indexed_partial": ([vp, vp, u8p, vp, vp, u8p, vp, vp, sz, ctypes.c_int64, vp], ctypes.c_int),
        "b3_verify_multiple_indexed_partial_dev": ([vp, vp, vp, vp, vp, vp, vp, vp, sz, ctypes.c_int64, vp], ctypes.c_int),
        "b3_nccl_unique_id": ([u8p], ctypes.c_int),
        "b3_comm_create": ([ctypes.c_int, ctypes.c_int, ctypes.c_int, u8p, ctypes.c_int, ctypes.POINTER(vp)], ctypes.c_int),
        "b3_comm_destroy": ([vp], None),
        "b3_comm_last_error": ([vp], ctypes.c_char_p),
        "b3_comm_collective_count": ([vp], ctypes.c_uint64),
        "b3_sharded_begin": ([vp, vp, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp, sz, ctypes.c_int64, ctypes.c_int, i64p], ctypes.c_int),
        "b3_sharded_finish": ([vp, vp, ctypes.c_int, ctypes.c_int64, ip, i64p, u8p], ctypes.c_int),
        "b3_verify_multiple_sharded": ([vp, vp, ctypes.c_int, vp, vp, vp, vp, vp, vp, vp, sz, ctypes.c_int64, ctypes.c_int, ip, i64p, u8p],
                                       ctypes.c_int),
        "b3_verify_batch": ([vp, ctypes.c_int, u8p, u8p, vp, u8p, vp, sz, i32p, i32p, u8p], ctypes.c_int),
        "b3_verify_batch_dev": ([vp, ctypes.c_int, vp, vp, vp, vp, vp, sz, vp, vp, vp], ctypes.c_int),
        "b3_verify_multiple_partial_dev": ([vp, vp, vp, vp, vp, vp, vp, sz, ctypes.c_int64, vp], ctypes.c_int),
        "b3_verify_multiple_partial": ([vp, u8p, u8p, vp, u8p, vp, vp, sz, ctypes.c_int64, vp], ctypes.c_int),
        "b3_combine_partials_dev": ([vp, vp, sz, ip, i64p, u8p], ctypes.c_int),
        "b3_hash_to_g2_dev": ([vp, vp, vp, sz, vp], ctypes.c_int),
        "b3_g1_aggregate_dev": ([vp, vp, vp, sz, vp, vp], ctypes.c_int),
        "b3_g1_mul_gen": ([vp, u8p, sz, u8p], ctypes.c_int),
        "b3_g2_mul": ([vp, u8p, u8p, sz, u8p], ctypes.c_int),
        "b3_imad_peak": ([vp, ctypes.c_int, ctypes.POINTER(ctypes.c_double)], ctypes.c_int),
    }
    for name, (args, res) in sigs.items():
        fn = getattr(L, name)          # AttributeError here = header/library mismatch: fail loudly
        fn.argtypes = args
        fn.restype = res
    L._b3_symbols = sorted(sigs)
    _lib = L
    return L


def _symbols_of_table():
    """Names bound above, read from this file's own source (so the list cannot drift from the table)."""
    import re
    src = open(os.path.abspath(__file__).replace(".pyc", ".py")).read()
    return sorted(set(re.findall(r'^        "(b3_[a-z0-9_]+)": \(', src, flags=re.M)))


EXPORTED_SYMBOLS = _symbols_of_table()
