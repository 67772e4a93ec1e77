"""Host-side mirror of the milagro_bls verification API over the C ABI (include/milagro_bls_b200.h).

Same names, argument meaning and error behaviour as the reference's Rust types (M = /root/reference/src):
  PublicKey               M/src/keys.rs:116-187        Signature            M/src/signature.rs:9-51
  AggregatePublicKey      M/src/aggregates.rs:17-78    AggregateSignature   M/src/aggregates.rs:83-334
Decoding errors raise AmclError(kind) (A/errors.rs:1-11); every verify* returns a plain bool.
A point is held as its ZCash *uncompressed* encoding (96 B for G1, 192 B for G2) -- the byte string the
reference's own serialize_uncompressed_g1/g2 produces -- so equality of objects is equality of group elements,
as with the reference's projective PartialEq (SURVEY.md C.8).

All arithmetic runs on the GPU through the C ABI.  There is no CPU path here.
"""
import ctypes
import threading

import numpy as np

from . import _lib
from .rng import draw_scalar

G1_BYTES, G2_BYTES = 48, 96
G1_INF = bytes([0x40]) + bytes(95)
G2_INF = bytes([0x40]) + bytes(191)


class AmclError(Exception):
    def __init__(self, kind):
        super().__init__(kind)
        self.kind = kind


def _raise(code, ctx=None):
    name = _lib.ERR_NAMES.get(code, f"error {code}")
    if code <= -100:
        msg = ""
        if ctx is not None and ctx.handle:
            msg = _lib.lib().b3_last_error(ctx.handle).decode(errors="replace")
        raise RuntimeError(f"milagro_bls_b200: {name} {msg}")
    raise AmclError(name)


def _buf(b):
    """bytes / bytearray / numpy uint8 array -> (void*, keepalive)"""
    if isinstance(b, np.ndarray):
        a = np.ascontiguousarray(b, dtype=np.uint8)
        return ctypes.c_void_p(a.ctypes.data), a
    a = np.frombuffer(bytes(b), dtype=np.uint8) if len(b) else np.zeros(1, dtype=np.uint8)
    return ctypes.c_void_p(a.ctypes.data), a


def _need(cond, what):
    """Argument validation before anything reaches the C side (which trusts its sizes)."""
    if not cond:
        raise ValueError(f"milagro_bls_b200: {what}")


def _u32(a):
    return np.ascontiguousarray(a, dtype=np.uint32)


def _offsets(chunks):
    off = np.zeros(len(chunks) + 1, dtype=np.uint32)
    if len(chunks):
        off[1:] = np.cumsum([len(c) for c in chunks], dtype=np.uint64).astype(np.uint32)
    return off


class Engine:
    """One CUDA context of the library (one per thread / per GPU)."""

    def __init__(self, device=0):
        self.L = _lib.lib()
        h = ctypes.c_void_p()
        rc = self.L.b3_ctx_create(int(device), ctypes.byref(h))
        self.handle = h if rc == 0 else None
        if rc != 0:
            raise RuntimeError(
                f"milagro_bls_b200: cannot create a context on CUDA device {device} (code {rc}); "
                "an sm_100 (B200) GPU is required -- there is no CPU fallback")
        self.device = device

    def close(self):
        if self.handle:
            self.L.b3_ctx_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- raw batched entry points (numpy in / numpy out) ------------------------------------------------
    def _ck(self, rc):
        if rc != 0:
            _raise(rc, self)

    @property
    def launches(self):
        return int(self.L.b3_ctx_launch_count(self.handle))

    def last_kernel_ms(self, which=0):
        return float(self.L.b3_ctx_last_kernel_ms(self.handle, which))

    def set_serial(self, serial=True):
        """serial=True: independent stages run one after another (per-stage timing); False: overlapped (default)."""
        self.L.b3_ctx_set_serial(self.handle, 1 if serial else 0)

    def set_item_kernel(self, which=0):
        """Finishing kernel of verify_batch: 0 = by batch size, 1 = CTA per item, 3 = lane pair per item."""
        self.L.b3_ctx_set_item_kernel(self.handle, int(which))

    def stage_ms(self):
        """{stage name: device ms} of the most recent verification / hash call (CUDA events on the library's stream)."""
        return {self.L.b3_stage_name(i).decode(): float(self.L.b3_ctx_stage_ms(self.handle, i)) for i in range(self.L.b3_stage_count())}

    def g1_decompress(self, data48, validate=True):
        n = len(data48) // 48
        p, keep = _buf(data48)
        out = np.zeros(96 * max(n, 1), dtype=np.uint8)
        st = np.zeros(max(n, 1), dtype=np.int32)
        self._ck(self.L.b3_g1_decompress(self.handle, p, n, 1 if validate else 0, out.ctypes.data,
                                         st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
        return out[:96 * n], st[:n]

    def g2_decompress(self, data96):
        n = len(data96) // 96
        p, keep = _buf(data96)
        out = np.zeros(192 * max(n, 1), dtype=np.uint8)
        st = np.zeros(max(n, 1), dtype=np.int32)
        self._ck(self.L.b3_g2_decompress(self.handle, p, n, out.ctypes.data, st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
        return out[:192 * n], st[:n]

    def g1_compress(self, data96):
        n = len(data96) // 96
        p, keep = _buf(data96)
        out = np.zeros(48 * max(n, 1), dtype=np.uint8)
        st = np.zeros(max(n, 1), dtype=np.int32)
        self._ck(self.L.b3_g1_compress(self.handle, p, n, out.ctypes.data, st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
        return out[:48 * n], st[:n]

    def g2_compress(self, data192):
        n = len(data192) // 192
        p, keep = _buf(data192)
        out = np.zeros(96 * max(n, 1), dtype=np.uint8)
        st = np.zeros(max(n, 1), dtype=np.int32)
        self._ck(self.L.b3_g2_compress(self.handle, p, n, out.ctypes.data, st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
        return out[:96 * n], st[:n]

    def g1_validate(self, data96):
        n = len(data96) // 96
        p, keep = _buf(data96)
        st = np.zeros(max(n, 1), dtype=np.int32)
        ok = np.zeros(max(n, 1), dtype=np.int32)
        i32 = ctypes.POINTER(ctypes.c_int32)
        self._ck(self.L.b3_g1_validate(self.handle, p, n, st.ctypes.data_as(i32), ok.ctypes.data_as(i32)))
        return st[:n], ok[:n]

    def g2_subgroup_check(self, data192):
        n = len(data192) // 192
        p, keep = _buf(data192)
        st = np.zeros(max(n, 1), dtype=np.int32)
        ok = np.zeros(max(n, 1), dtype=np.int32)
        i32 = ctypes.POINTER(ctypes.c_int32)
        self._ck(self.L.b3_g2_subgroup_check(self.handle, p, n, st.ctypes.data_as(i32), ok.ctypes.data_as(i32)))
        return st[:n], ok[:n]

    def g1_aggregate(self, pks96, offsets):
        off = np.ascontiguousarray(offsets, dtype=np.uint32)
        n = len(off) - 1
        _need(n >= 0 and (n == 0 or (off[0] == 0 and int(off[-1]) * 96 == len(pks96) and np.all(np.diff(off.astype(np.int64)) >= 0))),
              "g1_aggregate: offsets must start at 0, be non-decreasing and end at len(pks96) / 96")
        p, keep = _buf(pks96)
        out = np.zeros(96 * max(n, 1), dtype=np.uint8)
        st = np.zeros(max(n, 1), dtype=np.int32)
        self._ck(self.L.b3_g1_aggregate(self.handle, p, off.ctypes.data, n, out.ctypes.data,
                                        st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
        return out[:96 * n], st[:n]

    def g2_aggregate(self, sigs192, offsets):
        off = np.ascontiguousarray(offsets, dtype=np.uint32)
        n = len(off) - 1
        _need(n >= 0 and (n == 0 or (off[0] == 0 and int(off[-1]) * 192 == len(sigs192) and np.all(np.diff(off.astype(np.int64)) >= 0))),
              "g2_aggregate: offsets must start at 0, be non-decreasing and end at len(sigs192) / 192")
        p, keep = _buf(sigs192)
        out = np.zeros(192 * max(n, 1), dtype=np.uint8)
        st = np.zeros(max(n, 1), dtype=np.int32)
        self._ck(self.L.b3_g2_aggregate(self.handle, p, off.ctypes.data, n, out.ctypes.data,
                                        st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
        return out[:192 * n], st[:n]

    def hash_to_g2(self, msgs, dst=None):
        """msgs: list of bytes -> (n, 192) uint8 array of uncompressed G2 points (M/src/amcl_utils.rs:33-35)."""
        n = len(msgs)
        off = _offsets(msgs)
        p, keep = _buf(b"".join(msgs))
        out = np.zeros(192 * max(n, 1), dtype=np.uint8)
        if dst is None:
            dp, dl, keep2 = None, 0, None
        else:
            dp, keep2 = _buf(dst)
            dl = len(dst)
        self._ck(self.L.b3_hash_to_g2(self.handle, p, off.ctypes.data, n, dp, dl, out.ctypes.data))
        return out[:192 * n].reshape(n, 192)

    def hash_to_g2_blob(self, msgs_blob, msg_offsets, dst=None):
        """hash_to_g2 over a packed message blob + n + 1 offsets (no per-message Python objects)."""
        off = _u32(msg_offsets)
        n = len(off) - 1
        _need(n >= 0 and (n == 0 or (off[0] == 0 and int(off[-1]) == len(msgs_blob))), "hash_to_g2_blob: offsets must be n + 1 values ending at len(msgs)")
        p, keep = _buf(msgs_blob)
        out = np.zeros(192 * max(n, 1), dtype=np.uint8)
        if dst is None:
            dp, dl, keep2 = None, 0, None
        else:
            dp, keep2 = _buf(dst)
            dl = len(dst)
        self._ck(self.L.b3_hash_to_g2(self.handle, p, off.ctypes.data, n, dp, dl, out.ctypes.data))
        return out[:192 * n].reshape(n, 192)

    def verify(self, sig192, pk96, msg, want_gt=False):
        _need(len(sig192) == 192 and len(pk96) == 96, "verify: signature must be 192 bytes and the key 96 bytes (uncompressed)")
        ok = ctypes.c_int(0)
        gt = np.zeros(576, dtype=np.uint8)
        ps, k1 = _buf(sig192)
        pp, k2 = _buf(pk96)
        pm, k3 = _buf(msg)
        self._ck(self.L.b3_verify(self.handle, ps, pp, pm, len(msg), ctypes.byref(ok), gt.ctypes.data))
        return (bool(ok.value), gt.tobytes()) if want_gt else bool(ok.value)

    def fast_aggregate_verify(self, sig192, pks96, msg, want_gt=False):
        _need(len(sig192) == 192 and len(pks96) % 96 == 0, "fast_aggregate_verify: 192-byte signature, keys a multiple of 96 bytes")
        ok = ctypes.c_int(0)
        gt = np.zeros(576, dtype=np.uint8)
        ps, k1 = _buf(sig192)
        pp, k2 = _buf(pks96)
        pm, k3 = _buf(msg)
        self._ck(self.L.b3_fast_aggregate_verify(self.handle, ps, pp, len(pks96) // 96, pm, len(msg), ctypes.byref(ok), gt.ctypes.data))
        return (bool(ok.value), gt.tobytes()) if want_gt else bool(ok.value)

    def fast_aggregate_verify_pre_aggregated(self, sig192, apk96, msg, want_gt=False):
        _need(len(sig192) == 192 and len(apk96) == 96, "fast_aggregate_verify_pre_aggregated: 192-byte signature, 96-byte key")
        ok = ctypes.c_int(0)
        gt = np.zeros(576, dtype=np.uint8)
        ps, k1 = _buf(sig192)
        pp, k2 = _buf(apk96)
        pm, k3 = _buf(msg)
        self._ck(self.L.b3_fast_aggregate_verify_pre_aggregated(self.handle, ps, pp, pm, len(msg), ctypes.byref(ok), gt.ctypes.data))
        return (bool(ok.value), gt.tobytes()) if want_gt else bool(ok.value)

    def aggregate_verify(self, sig192, pks96, msgs, want_gt=False):
        ok = ctypes.c_int(0)
        gt = np.zeros(576, dtype=np.uint8)
        n = len(msgs)
        _need(len(sig192) == 192 and len(pks96) == 96 * n, "aggregate_verify: 192-byte signature and one 96-byte key per message")
        off = _offsets(msgs)
        ps, k1 = _buf(sig192)
        pp, k2 = _buf(pks96)
        pm, k3 = _buf(b"".join(msgs))
        self._ck(self.L.b3_aggregate_verify(self.handle, ps, pp, pm, off.ctypes.data, n, ctypes.byref(ok), gt.ctypes.data))
        return (bool(ok.value), gt.tobytes()) if want_gt else bool(ok.value)

    def _vm_args(self, sigs192, keys, key_bytes, pk_offsets, msgs_blob, msg_offsets, scalars, what):
        """Validated, contiguous arguments of a verify_multiple-shaped call.  keys: bytes / uint8 array of 96-byte records
        (key_bytes = 96) or an array of u32 table indices (key_bytes = 4)."""
        sc = np.ascontiguousarray(scalars, dtype=np.uint64)
        n = len(sc)
        moff = _u32(msg_offsets)
        _need(len(moff) == n + 1 and (n == 0 or moff[0] == 0) and int(moff[-1]) == len(msgs_blob), f"{what}: message offsets must be n + 1 values ending at len(msgs)")
        _need(sigs192 is None or len(sigs192) == 192 * n, f"{what}: one 192-byte signature per set")
        if key_bytes == 4:
            kk = _u32(keys)
            nk = len(kk)
            pp, k2 = ctypes.c_void_p(kk.ctypes.data), kk
        else:
            _need(len(keys) % 96 == 0, f"{what}: keys must be 96-byte records")
            nk = len(keys) // 96
            pp, k2 = _buf(keys)
        if pk_offsets is None:
            _need(nk == n, f"{what}: one key per set when pk_offsets is None")
            koff, po = None, None
        else:
            koff = _u32(pk_offsets)
            _need(len(koff) == n + 1 and (n == 0 or koff[0] == 0) and int(koff[-1]) == nk and np.all(np.diff(koff.astype(np.int64)) >= 0),
                  f"{what}: key offsets must be n + 1 non-decreasing values ending at the number of keys")
            po = koff.ctypes.data
        ps, k1 = (None, None) if sigs192 is None else _buf(sigs192)
        pm, k3 = _buf(msgs_blob)
        return n, ps, pp, po, pm, moff, sc, (k1, k2, k3, koff)

    def verify_multiple(self, sigs192, pks96, pk_offsets, msgs_blob, msg_offsets, scalars, want_gt=False):
        """Raw batched form of verify_multiple_aggregate_signatures.  pk_offsets None -> pks96 holds one
        (aggregate) key per set.  Returns (accept, first_bad[, gt])."""
        n, ps, pp, po, pm, moff, sc, keep = self._vm_args(sigs192, pks96, 96, pk_offsets, msgs_blob, msg_offsets, scalars, "verify_multiple")
        ok = ctypes.c_int(0)
        fb = ctypes.c_int64(-1)
        gt = np.zeros(576, dtype=np.uint8)
        self._ck(self.L.b3_verify_multiple(self.handle, ps, pp, po, pm, moff.ctypes.data, sc.ctypes.data, n,
                                           ctypes.byref(ok), ctypes.byref(fb), gt.ctypes.data))
        return (bool(ok.value), int(fb.value), gt.tobytes()) if want_gt else (bool(ok.value), int(fb.value))

    def verify_multiple_dev(self, table, d_sigs, d_keys, d_pk_off, d_msgs, d_msg_off, d_scalars, n, want_gt=False):
        """The whole call on inputs resident in HBM (device pointers as integers).  table None: d_keys = 96-byte records
        (b3_verify_multiple_dev); else u32 indices into the table (b3_verify_multiple_indexed_dev).  Returns (accept, first_bad[, gt])."""
        ok = ctypes.c_int(0)
        fb = ctypes.c_int64(-1)
        gt = np.zeros(576, dtype=np.uint8)
        if table is None:
            self._ck(self.L.b3_verify_multiple_dev(self.handle, d_sigs, d_keys, d_pk_off, d_msgs, d_msg_off, d_scalars, n,
                                                   ctypes.byref(ok), ctypes.byref(fb), gt.ctypes.data))
        else:
            self._ck(self.L.b3_verify_multiple_indexed_dev(self.handle, table.handle, d_sigs, d_keys, d_pk_off, d_msgs, d_msg_off, d_scalars, n,
                                                           ctypes.byref(ok), ctypes.byref(fb), gt.ctypes.data))
        return (bool(ok.value), int(fb.value), gt.tobytes()) if want_gt else (bool(ok.value), int(fb.value))

    def verify_multiple_grouped(self, table, sigs192, keys, pk_offsets, msgs_blob, msg_offsets, msg_idx, scalars, want_gt=False):
        """verify_multiple over sets that name their message by index: set j signs message msg_idx[j], message k is
        msgs_blob[msg_offsets[k]:msg_offsets[k + 1]].  Each distinct message is hashed and paired once; the result equals
        verify_multiple / verify_multiple_indexed on the expanded inputs.  table None: keys = 96-byte records, else u32 indices
        into the KeyTable.  sigs192 None -> the signatures of the preceding sig_precheck.  Returns (accept, first_bad[, gt])."""
        sc = np.ascontiguousarray(scalars, dtype=np.uint64)
        n = len(sc)
        mi = _u32(msg_idx)
        moff = _u32(msg_offsets)
        n_msgs = len(moff) - 1
        _need(len(mi) == n, "verify_multiple_grouped: one message index per set")
        _need(n_msgs >= 0 and moff[0] == 0 and int(moff[-1]) == len(msgs_blob),
              "verify_multiple_grouped: message offsets must be n_msgs + 1 values ending at len(msgs)")
        # the set-shaped checks of _vm_args on a one-message-per-set stand-in of the offsets
        _, ps, pp, po, pm, _, sc, keep = self._vm_args(sigs192, keys, 96 if table is None else 4, pk_offsets, msgs_blob,
                                                       np.array([0] * n + [len(msgs_blob)], dtype=np.uint32), sc, "verify_multiple_grouped")
        ok = ctypes.c_int(0)
        fb = ctypes.c_int64(-1)
        gt = np.zeros(576, dtype=np.uint8)
        self._ck(self.L.b3_verify_multiple_grouped(self.handle, None if table is None else table.handle, ps, pp, po, pm, moff.ctypes.data,
                                                   max(n_msgs, 0), mi.ctypes.data, sc.ctypes.data, n, 0, ctypes.byref(ok), ctypes.byref(fb),
                                                   gt.ctypes.data))
        return (bool(ok.value), int(fb.value), gt.tobytes()) if want_gt else (bool(ok.value), int(fb.value))

    def verify_multiple_grouped_dev(self, table, d_sigs, d_keys, d_pk_off, d_msgs, d_msg_off, n_msgs, d_msg_idx, d_scalars, n, want_gt=False):
        """verify_multiple_grouped on inputs resident in HBM (device pointers as integers).  Returns (accept, first_bad[, gt])."""
        ok = ctypes.c_int(0)
        fb = ctypes.c_int64(-1)
        gt = np.zeros(576, dtype=np.uint8)
        self._ck(self.L.b3_verify_multiple_grouped(self.handle, None if table is None else table.handle, d_sigs, d_keys, d_pk_off, d_msgs,
                                                   d_msg_off, int(n_msgs), d_msg_idx, d_scalars, int(n), 1, ctypes.byref(ok), ctypes.byref(fb),
                                                   gt.ctypes.data))
        return (bool(ok.value), int(fb.value), gt.tobytes()) if want_gt else (bool(ok.value), int(fb.value))

    def verify_multiple_locate(self, n):
        """Per-set verdicts of the preceding whole verify_multiple call on this engine (verify_multiple, _checked, _indexed,
        _dev forms) that returned without raising: bool array, True where set j alone passes verify_multiple.  Any other call
        in between, or a different n, raises RuntimeError (BadArgument)."""
        valid = np.zeros(max(int(n), 1), dtype=np.int32)
        n_bad = ctypes.c_size_t(0)
        self._ck(self.L.b3_verify_multiple_locate(self.handle, int(n), valid.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), ctypes.byref(n_bad)))
        return valid[:n].astype(bool)

    def sig_precheck(self, sigs192):
        """Phase one of the two-phase call: upload, parse and subgroup-check the signatures; returns first_bad (-1: all passed).
        The checked signatures stay in this context for verify_multiple_checked / verify_multiple_indexed(sigs192=None)."""
        _need(len(sigs192) % 192 == 0, "sig_precheck: signatures must be 192-byte records")
        fb = ctypes.c_int64(-1)
        ps, k1 = _buf(sigs192)
        self._ck(self.L.b3_sig_precheck(self.handle, ps, len(sigs192) // 192, ctypes.byref(fb)))
        return int(fb.value)

    def verify_multiple_checked(self, pks96, pk_offsets, msgs_blob, msg_offsets, scalars, want_gt=False):
        """Phase two: the batch equation over the signatures of the preceding sig_precheck.  Returns accept[, gt]."""
        n, ps, pp, po, pm, moff, sc, keep = self._vm_args(None, pks96, 96, pk_offsets, msgs_blob, msg_offsets, scalars, "verify_multiple_checked")
        ok = ctypes.c_int(0)
        gt = np.zeros(576, dtype=np.uint8)
        self._ck(self.L.b3_verify_multiple_checked(self.handle, pp, po, pm, moff.ctypes.data, sc.ctypes.data, n, ctypes.byref(ok), gt.ctypes.data))
        return (bool(ok.value), gt.tobytes()) if want_gt else bool(ok.value)

    def verify_multiple_indexed(self, table, sigs192, key_idx, pk_offsets, msgs_blob, msg_offsets, scalars, want_gt=False):
        """verify_multiple with the keys named by u32 indices into a KeyTable.  sigs192 None -> the signatures of the
        preceding sig_precheck.  Returns (accept, first_bad[, gt])."""
        n, ps, pp, po, pm, moff, sc, keep = self._vm_args(sigs192, key_idx, 4, pk_offsets, msgs_blob, msg_offsets, scalars, "verify_multiple_indexed")
        ok = ctypes.c_int(0)
        fb = ctypes.c_int64(-1)
        gt = np.zeros(576, dtype=np.uint8)
        self._ck(self.L.b3_verify_multiple_indexed(self.handle, table.handle, ps, pp, po, pm, moff.ctypes.data, sc.ctypes.data, n,
                                                   ctypes.byref(ok), ctypes.byref(fb), gt.ctypes.data))
        return (bool(ok.value), int(fb.value), gt.tobytes()) if want_gt else (bool(ok.value), int(fb.value))

    def g1_aggregate_indexed(self, table, key_idx, offsets):
        off = _u32(offsets)
        kk = _u32(key_idx)
        n = len(off) - 1
        _need(n >= 0 and (n == 0 or (off[0] == 0 and int(off[-1]) == len(kk) and np.all(np.diff(off.astype(np.int64)) >= 0))),
              "g1_aggregate_indexed: offsets must start at 0, be non-decreasing and end at len(key_idx)")
        out = np.zeros(96 * max(n, 1), dtype=np.uint8)
        st = np.zeros(max(n, 1), dtype=np.int32)
        self._ck(self.L.b3_g1_aggregate_indexed(self.handle, table.handle, kk.ctypes.data, off.ctypes.data, n, out.ctypes.data,
                                                st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
        return out[:96 * n], st[:n]

    def set_latency_mode(self, mode=0):
        """Chain kernels of verify_multiple: 0 = replicated lanes when the call is alone on its GPU (default), 1 = always, 2 = never."""
        self.L.b3_ctx_set_latency_mode(self.handle, int(mode))

    def set_trusted_points(self, trusted=True):
        """trusted=True: the point arrays passed to this context come out of this library's own decompress / validate calls
        (the reference's type invariant), so the aggregation kernels skip their on-curve checks."""
        self.L.b3_ctx_set_trusted_points(self.handle, 1 if trusted else 0)

    def verify_batch(self, mode, sigs192, pks96, pk_offsets, msgs, want_gt=False):
        """n independent items, one accept bit each (b3_verify_batch).  mode: _lib.ITEM_VERIFY (one key per item),
        ITEM_FAST_AGGREGATE (keys of item i = pks96[pk_offsets[i]:pk_offsets[i+1]]), ITEM_PRE_AGGREGATED.
        msgs: list of byte strings.  Returns (accept[n] bool array, status[n] int32 array[, gt (n, 576) uint8])."""
        n = len(msgs)
        _need(len(sigs192) == 192 * n and len(pks96) % 96 == 0, "verify_batch: one 192-byte signature per item, keys in 96-byte records")
        if pk_offsets is None:
            _need(len(pks96) == 96 * n, "verify_batch: one key per item when pk_offsets is None")
        else:
            ko = _u32(pk_offsets)
            _need(len(ko) == n + 1 and (n == 0 or ko[0] == 0) and int(ko[-1]) * 96 == len(pks96) and np.all(np.diff(ko.astype(np.int64)) >= 0),
                  "verify_batch: key offsets must be n + 1 non-decreasing values ending at the number of keys")
        accept = np.zeros(max(n, 1), dtype=np.int32)
        status = np.zeros(max(n, 1), dtype=np.int32)
        gt = np.zeros((max(n, 1), 576), dtype=np.uint8) if want_gt else None
        off = _offsets(msgs)
        ps, k1 = _buf(sigs192)
        pp, k2 = _buf(pks96)
        pm, k3 = _buf(b"".join(msgs))
        po = None
        if pk_offsets is not None:
            koff = np.ascontiguousarray(pk_offsets, dtype=np.uint32)
            po = koff.ctypes.data
        self._ck(self.L.b3_verify_batch(self.handle, mode, ps, pp, po, pm, off.ctypes.data, n,
                                        accept.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                        status.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)),
                                        gt.ctypes.data if want_gt else None))
        res = (accept[:n].astype(bool), status[:n])
        return res + (gt[:n],) if want_gt else res

    def verify_batch_dev(self, mode, d_sigs, d_pks, d_pk_off, d_msgs, d_msg_off, n, d_accept, d_status, d_gt=None):
        self._ck(self.L.b3_verify_batch_dev(self.handle, mode, d_sigs, d_pks, d_pk_off, d_msgs, d_msg_off, n, d_accept, d_status, d_gt))

    # device-pointer forms (torch tensors / raw addresses), used by bench.py and the multi-GPU path
    def verify_multiple_partial_dev(self, d_sigs, d_pks, d_pk_off, d_msgs, d_msg_off, d_scalars, n, index_base, d_partial):
        self._ck(self.L.b3_verify_multiple_partial_dev(self.handle, d_sigs, d_pks, d_pk_off, d_msgs, d_msg_off, d_scalars, n,
                                                       index_base, d_partial))

    def verify_multiple_partial(self, sigs192, pks96, pk_offsets, msgs_blob, msg_offsets, scalars, index_base, d_partial):
        """This rank's shard from HOST buffers -> 592-byte partial in device memory at d_partial (b3_verify_multiple_partial)."""
        n, ps, pp, po, pm, moff, sc, keep = self._vm_args(sigs192, pks96, 96, pk_offsets, msgs_blob, msg_offsets, scalars, "verify_multiple_partial")
        self._ck(self.L.b3_verify_multiple_partial(self.handle, ps, pp, po, pm, moff.ctypes.data, sc.ctypes.data, n, index_base, d_partial))

    def verify_multiple_indexed_partial(self, table, sigs192, key_idx, pk_offsets, msgs_blob, msg_offsets, scalars, index_base, d_partial):
        n, ps, pp, po, pm, moff, sc, keep = self._vm_args(sigs192, key_idx, 4, pk_offsets, msgs_blob, msg_offsets, scalars,
                                                          "verify_multiple_indexed_partial")
        self._ck(self.L.b3_verify_multiple_indexed_partial(self.handle, table.handle, ps, pp, po, pm, moff.ctypes.data, sc.ctypes.data, n,
                                                           index_base, d_partial))

    def verify_multiple_indexed_partial_dev(self, table, d_sigs, d_idx, d_pk_off, d_msgs, d_msg_off, d_scalars, n, index_base, d_partial):
        self._ck(self.L.b3_verify_multiple_indexed_partial_dev(self.handle, table.handle, d_sigs, d_idx, d_pk_off, d_msgs, d_msg_off, d_scalars, n,
                                                               index_base, d_partial))

    # ---- multi-GPU (b3_comm_*: NCCL behind the C ABI) ---------------------------------------------------------
    def sharded_begin(self, comm, lane, table, sigs192, keys, pk_offsets, msgs_blob, msg_offsets, scalars, index_base):
        """This rank's shard (HOST buffers) -> partial, deposited for the step's all-gather.  keys: 96-byte records (table None) or
        u32 table indices.  Returns the ticket for sharded_finish."""
        n, ps, pp, po, pm, moff, sc, keep = self._vm_args(sigs192, keys, 96 if table is None else 4, pk_offsets, msgs_blob, msg_offsets, scalars,
                                                          "sharded_begin")
        t = ctypes.c_int64(-1)
        self._ck(self.L.b3_sharded_begin(self.handle, comm.handle, lane, None if table is None else table.handle, ps, pp, po, pm,
                                         moff.ctypes.data, sc.ctypes.data, n, index_base, 0, ctypes.byref(t)))
        return int(t.value)

    def sharded_begin_dev(self, comm, lane, table, d_sigs, d_keys, d_pk_off, d_msgs, d_msg_off, d_scalars, n, index_base):
        t = ctypes.c_int64(-1)
        self._ck(self.L.b3_sharded_begin(self.handle, comm.handle, lane, None if table is None else table.handle, d_sigs, d_keys, d_pk_off,
                                         d_msgs, d_msg_off, d_scalars, n, index_base, 1, ctypes.byref(t)))
        return int(t.value)

    def sharded_finish(self, comm, lane, ticket, want_gt=False):
        ok = ctypes.c_int(0)
        fb = ctypes.c_int64(-1)
        gt = np.zeros(576, dtype=np.uint8)
        self._ck(self.L.b3_sharded_finish(self.handle, comm.handle, lane, ticket, ctypes.byref(ok), ctypes.byref(fb), gt.ctypes.data))
        return (bool(ok.value), int(fb.value), gt.tobytes()) if want_gt else (bool(ok.value), int(fb.value))

    def combine_partials_dev(self, d_partials, n_partials, want_gt=False):
        ok = ctypes.c_int(0)
        fb = ctypes.c_int64(-1)
        gt = np.zeros(576, dtype=np.uint8)
        self._ck(self.L.b3_combine_partials_dev(self.handle, d_partials, n_partials, ctypes.byref(ok), ctypes.byref(fb), gt.ctypes.data))
        return (bool(ok.value), int(fb.value), gt.tobytes()) if want_gt else (bool(ok.value), int(fb.value))

    def hash_to_g2_dev(self, d_msgs, d_off, n, d_out):
        self._ck(self.L.b3_hash_to_g2_dev(self.handle, d_msgs, d_off, n, d_out))

    def g1_aggregate_dev(self, d_pks, d_off, n_sets, d_out, d_status):
        self._ck(self.L.b3_g1_aggregate_dev(self.handle, d_pks, d_off, n_sets, d_out, d_status))

    # signing-side helpers (input synthesis only)
    def g1_mul_gen(self, scalars):
        n = len(scalars)
        blob = b"".join(int(s).to_bytes(32, "big") for s in scalars)
        p, keep = _buf(blob)
        out = np.zeros(96 * max(n, 1), dtype=np.uint8)
        self._ck(self.L.b3_g1_mul_gen(self.handle, p, n, out.ctypes.data))
        return out[:96 * n].reshape(n, 96)

    def g2_mul(self, pts192, scalars):
        n = len(scalars)
        blob = b"".join(int(s).to_bytes(32, "big") for s in scalars)
        pp, k1 = _buf(pts192)
        p, keep = _buf(blob)
        out = np.zeros(192 * max(n, 1), dtype=np.uint8)
        self._ck(self.L.b3_g2_mul(self.handle, pp, p, n, out.ctypes.data))
        return out[:192 * n].reshape(n, 192)

    def imad_peak(self, wide=False):
        v = ctypes.c_double(0)
        self._ck(self.L.b3_imad_peak(self.handle, 1 if wide else 0, ctypes.byref(v)))
        return v.value


class KeyTable:
    """Device-resident table of decoded public keys (b3_keytable_*): PublicKey::from_bytes -- decompression + key_validate,
    M/src/keys.rs:140-147 -- paid once per validator; verification names keys by index.  Shared by every Engine of its device."""

    def __init__(self, engine, capacity=0):
        self.L = engine.L
        self.engine = engine
        h = ctypes.c_void_p()
        engine._ck(self.L.b3_keytable_create(engine.handle, int(capacity), ctypes.byref(h)))
        self.handle = h

    def __len__(self):
        return int(self.L.b3_keytable_size(self.handle))

    def append(self, keys, compressed=True, validate=True):
        """keys: bytes / uint8 array of 48-byte compressed (compressed=True) or 96-byte uncompressed records.
        Returns (first_index, status[n])."""
        rec = 48 if compressed else 96
        _need(len(keys) % rec == 0, f"KeyTable.append: keys must be {rec}-byte records")
        n = len(keys) // rec
        p, keep = _buf(keys)
        st = np.zeros(max(n, 1), dtype=np.int32)
        first = ctypes.c_size_t(0)
        self.engine._ck(self.L.b3_keytable_append(self.engine.handle, self.handle, p, n, 1 if compressed else 0, 1 if validate else 0,
                                                  st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), ctypes.byref(first)))
        return int(first.value), st[:n]

    def get(self, idx):
        kk = _u32(idx)
        n = len(kk)
        out = np.zeros(96 * max(n, 1), dtype=np.uint8)
        st = np.zeros(max(n, 1), dtype=np.int32)
        self.engine._ck(self.L.b3_keytable_get(self.engine.handle, self.handle, kk.ctypes.data, n, out.ctypes.data,
                                               st.ctypes.data_as(ctypes.POINTER(ctypes.c_int32))))
        return out[:96 * n].reshape(n, 96), st[:n]

    def close(self):
        if self.handle:
            self.L.b3_keytable_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def nccl_unique_id():
    """128-byte NCCL unique id (call on one rank, ship to the others by any transport)."""
    buf = np.zeros(128, dtype=np.uint8)
    rc = _lib.lib().b3_nccl_unique_id(buf.ctypes.data)
    if rc != 0:
        raise RuntimeError("milagro_bls_b200: NCCL not available (libnccl.so.2 could not be bound)")
    return buf.tobytes()


class Comm:
    """b3_comm: one NCCL communicator serving `lanes` contexts of this process (see include/milagro_bls_b200.h)."""

    def __init__(self, device, nranks, rank, unique_id, lanes=1):
        self.L = _lib.lib()
        h = ctypes.c_void_p()
        idb = np.frombuffer(bytes(unique_id), dtype=np.uint8).copy() if unique_id is not None else None
        rc = self.L.b3_comm_create(int(device), int(nranks), int(rank), None if idb is None else idb.ctypes.data, int(lanes), ctypes.byref(h))
        if rc != 0:
            raise RuntimeError(f"milagro_bls_b200: b3_comm_create failed (code {rc})")
        self.handle = h
        self.nranks, self.rank, self.lanes = nranks, rank, lanes

    @property
    def collectives(self):
        return int(self.L.b3_comm_collective_count(self.handle))

    def close(self):
        if self.handle:
            self.L.b3_comm_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


_default = threading.local()


def default_engine():
    e = getattr(_default, "engine", None)
    if e is None:
        e = Engine(0)
        _default.engine = e
    return e


def set_default_engine(e):
    _default.engine = e


# ---------------------------------------------------------------------------------------------------------
# Reference-shaped types
# ---------------------------------------------------------------------------------------------------------
class PublicKey:
    """M/src/keys.rs:116-187.  `point`: 96-byte uncompressed encoding."""
    __slots__ = ("point",)

    def __init__(self, point):
        self.point = bytes(point)
        _need(len(self.point) == 96, "PublicKey.point is the 96-byte uncompressed encoding")

    @staticmethod
    def from_bytes(data, engine=None):                       # keys.rs:140-147 (validates)
        return PublicKey._decode(data, True, engine)

    @staticmethod
    def from_bytes_unchecked(data, engine=None):             # keys.rs:150-155
        return PublicKey._decode(data, False, engine)

    @staticmethod
    def _decode(data, validate, engine):
        data = bytes(data)
        if len(data) != G1_BYTES:                            # M/src/amcl_utils.rs:52-58
            raise AmclError("InvalidG1Size")
        e = engine or default_engine()
        out, st = e.g1_decompress(data, validate)
        if st[0]:
            _raise(int(st[0]))
        return PublicKey(out.tobytes())

    @staticmethod
    def from_uncompressed_bytes(data, engine=None):          # keys.rs:168-175
        data = bytes(data)
        if len(data) != 2 * G1_BYTES:
            raise AmclError("InvalidG1Size")
        e = engine or default_engine()
        st, _ = e.g1_validate(data)
        if st[0]:
            _raise(int(st[0]))
        return PublicKey(data)

    def as_bytes(self, engine=None):                         # keys.rs:158-160
        e = engine or default_engine()
        out, st = e.g1_compress(self.point)
        if st[0]:
            _raise(int(st[0]))
        return out.tobytes()

    def as_uncompressed_bytes(self):                         # keys.rs:163-165
        return self.point

    def key_validate(self, engine=None):                     # keys.rs:181-186
        e = engine or default_engine()
        st, ok = e.g1_validate(self.point)
        return st[0] == 0 and bool(ok[0])

    def __eq__(self, o):
        return isinstance(o, PublicKey) and self.point == o.point

    def __hash__(self):
        return hash(self.point)


class AggregatePublicKey:
    """M/src/aggregates.rs:17-78."""
    __slots__ = ("point",)

    def __init__(self, point=G1_INF):
        self.point = bytes(point)
        _need(len(self.point) == 96, "AggregatePublicKey.point is the 96-byte uncompressed encoding")

    @staticmethod
    def aggregate(keys, engine=None):                        # aggregates.rs:29-39
        return AggregatePublicKey.into_aggregate(keys, engine)

    @staticmethod
    def into_aggregate(keys, engine=None):                   # aggregates.rs:46-56
        if len(keys) == 0:
            raise AmclError("AggregateEmptyPoints")
        e = engine or default_engine()
        blob = b"".join(k.point for k in keys)
        out, st = e.g1_aggregate(blob, [0, len(keys)])
        if st[0]:
            _raise(int(st[0]))
        return AggregatePublicKey(out.tobytes())

    @staticmethod
    def from_public_key(key):                                # aggregates.rs:61-63
        return AggregatePublicKey(key.point)

    def add(self, public_key, engine=None):                  # aggregates.rs:68-70
        e = engine or default_engine()
        out, st = e.g1_aggregate(self.point + public_key.point, [0, 2])
        if st[0]:
            _raise(int(st[0]))
        self.point = out.tobytes()

    def add_aggregate(self, other, engine=None):             # aggregates.rs:73-77
        self.add(other, engine)

    def __eq__(self, o):
        return isinstance(o, AggregatePublicKey) and self.point == o.point

    def __hash__(self):
        return hash(self.point)


class Signature:
    """M/src/signature.rs:9-51 (verification half; Signature::new needs a secret key and is out of scope)."""
    __slots__ = ("point",)

    def __init__(self, point):
        self.point = bytes(point)
        _need(len(self.point) == 192, "Signature.point is the 192-byte uncompressed encoding")

    @staticmethod
    def from_bytes(data, engine=None):                       # signature.rs:43-46 (no subgroup check)
        data = bytes(data)
        if len(data) != G2_BYTES:                            # M/src/amcl_utils.rs:68-74
            raise AmclError("InvalidG2Size")
        e = engine or default_engine()
        out, st = e.g2_decompress(data)
        if st[0]:
            _raise(int(st[0]))
        return Signature(out.tobytes())

    def as_bytes(self, engine=None):                         # signature.rs:49-51
        e = engine or default_engine()
        out, st = e.g2_compress(self.point)
        if st[0]:
            _raise(int(st[0]))
        return out.tobytes()

    def verify(self, msg, pk, engine=None):                  # signature.rs:27-40
        e = engine or default_engine()
        return e.verify(self.point, pk.point, bytes(msg))

    def __eq__(self, o):
        return isinstance(o, Signature) and self.point == o.point

    def __hash__(self):
        return hash(self.point)


class AggregateSignature:
    """M/src/aggregates.rs:83-334."""
    __slots__ = ("point",)

    def __init__(self, point=G2_INF):                        # AggregateSignature::new, aggregates.rs:93-95
        self.point = bytes(point)
        _need(len(self.point) == 192, "AggregateSignature.point is the 192-byte uncompressed encoding")

    @staticmethod
    def aggregate(signatures, engine=None):                  # aggregates.rs:100-106
        if len(signatures) == 0:
            return AggregateSignature()
        e = engine or default_engine()
        out, st = e.g2_aggregate(b"".join(s.point for s in signatures), [0, len(signatures)])
        if st[0]:
            _raise(int(st[0]))
        return AggregateSignature(out.tobytes())

    @staticmethod
    def from_signature(signature):                           # aggregates.rs:109-111
        return AggregateSignature(signature.point)

    def add(self, signature, engine=None):                   # aggregates.rs:114-116
        e = engine or default_engine()
        out, st = e.g2_aggregate(self.point + signature.point, [0, 2])
        if st[0]:
            _raise(int(st[0]))
        self.point = out.tobytes()

    def add_aggregate(self, other, engine=None):             # aggregates.rs:119-123
        self.add(other, engine)

    @staticmethod
    def from_bytes(data, engine=None):                       # aggregates.rs:319-322
        return AggregateSignature(Signature.from_bytes(data, engine).point)

    def as_bytes(self, engine=None):                         # aggregates.rs:325-327
        return Signature(self.point).as_bytes(engine)

    def aggregate_verify(self, msgs, public_keys, engine=None):               # aggregates.rs:130-170
        if len(msgs) != len(public_keys) or len(public_keys) == 0:
            return False
        e = engine or default_engine()
        return e.aggregate_verify(self.point, b"".join(k.point for k in public_keys), [bytes(m) for m in msgs])

    def fast_aggregate_verify(self, msg, public_keys, engine=None):           # aggregates.rs:177-215
        if len(public_keys) == 0:
            return False
        e = engine or default_engine()
        return e.fast_aggregate_verify(self.point, b"".join(k.point for k in public_keys), bytes(msg))

    def fast_aggregate_verify_pre_aggregated(self, msg, aggregate_public_key, engine=None):   # aggregates.rs:223-253
        e = engine or default_engine()
        return e.fast_aggregate_verify_pre_aggregated(self.point, aggregate_public_key.point, bytes(msg))

    @staticmethod
    def verify_multiple_aggregate_signatures(rng, signature_sets, engine=None):               # aggregates.rs:261-316
        """signature_sets: iterable of (AggregateSignature, AggregatePublicKey, msg bytes).
        `rng`: object with fill(n) -> bytes.  RNG consumption is bit-exact with the reference: one draw per set,
        in order, and none for / after the first set whose signature fails the subgroup check."""
        e = engine or default_engine()
        sets = list(signature_sets)
        n = len(sets)
        if n == 0:
            return True
        sigs = b"".join(s.point for s, _, _ in sets)
        # phase one (b3_sig_precheck): parse + subgroup-check every signature ONCE; they stay in the context for phase two
        try:
            first_bad = e.sig_precheck(sigs)
        except AmclError:
            raise
        n_draw = first_bad if first_bad >= 0 else n
        scalars = [draw_scalar(rng) for _ in range(n_draw)]
        if first_bad >= 0:
            return False
        msgs = [bytes(m) for _, _, m in sets]
        accept = e.verify_multiple_checked(b"".join(k.point for _, k, _ in sets), None, b"".join(msgs), _offsets(msgs),
                                           np.array(scalars, dtype=np.uint64))
        return accept

    @staticmethod
    def verify_multiple_aggregate_signatures_grouped(rng, signature_sets, engine=None):
        """Extension (the reference has no such function): verify_multiple_aggregate_signatures with every DISTINCT message
        hashed and paired once (Engine.verify_multiple_grouped), for batches whose sets repeat messages.  Messages are
        deduplicated by their bytes.  Result and RNG consumption are always those of verify_multiple_aggregate_signatures."""
        e = engine or default_engine()
        sets = list(signature_sets)
        n = len(sets)
        if n == 0:
            return True
        first_bad = e.sig_precheck(b"".join(s.point for s, _, _ in sets))
        n_draw = first_bad if first_bad >= 0 else n
        scalars = [draw_scalar(rng) for _ in range(n_draw)]
        if first_bad >= 0:
            return False
        index, msgs, msg_idx = {}, [], []
        for _, _, m in sets:
            m = bytes(m)
            if m not in index:
                index[m] = len(msgs)
                msgs.append(m)
            msg_idx.append(index[m])
        accept, _ = e.verify_multiple_grouped(None, None, b"".join(k.point for _, k, _ in sets), None, b"".join(msgs), _offsets(msgs),
                                              np.array(msg_idx, dtype=np.uint32), np.array(scalars, dtype=np.uint64))
        return accept

    @staticmethod
    def verify_multiple_aggregate_signatures_per_set(rng, signature_sets, engine=None):
        """Extension (the reference has no such function): one verdict per set, True where the set alone passes
        verify_multiple_aggregate_signatures.  signature_sets as there.  Exactly one scalar is drawn per set, in order, for
        every set -- there is no stop at the first bad set, since every set gets a verdict.  One batch call; if it rejects,
        the sets are located from what it left on the device (Engine.verify_multiple_locate).  Malformed points raise
        AmclError."""
        e = engine or default_engine()
        sets = list(signature_sets)
        n = len(sets)
        scalars = np.array([draw_scalar(rng) for _ in range(n)], dtype=np.uint64)
        if n == 0:
            return []
        msgs = [bytes(m) for _, _, m in sets]
        accept, _ = e.verify_multiple(b"".join(s.point for s, _, _ in sets), b"".join(k.point for _, k, _ in sets), None, b"".join(msgs),
                                      _offsets(msgs), scalars)
        if accept:
            return [True] * n
        return [bool(v) for v in e.verify_multiple_locate(n)]

    def __eq__(self, o):
        return isinstance(o, AggregateSignature) and self.point == o.point

    def __hash__(self):
        return hash(self.point)
