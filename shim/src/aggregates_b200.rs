//! Replacement bodies for `impl AggregatePublicKey` / `impl AggregateSignature` in the reference's src/aggregates.rs.
//! The struct definitions (one public field `point`, aggregates.rs:17-21, 83-87), `new`, `from_public_key`,
//! `from_signature`, `add`, `add_aggregate` (single point additions, aggregates.rs:61-77, 93-124) stay as they are.
use crate::aggregates::{AggregatePublicKey, AggregateSignature};
use crate::amcl_utils::{AmclError, G2_BYTES};
use crate::b200::ctx::{with_ctx, KeyTable};
use crate::b200::ffi::*;
use crate::b200::wire::*;
use crate::keys::PublicKey;
use crate::signature::Signature;
use rand::Rng;

/// One batch scalar, exactly as aggregates.rs:278-287 draws it: 8 bytes from the caller's RNG, i64::from_be_bytes(..).abs(),
/// retry while 0.  (i64::MIN, whose abs() overflows -- a panic in the reference's debug builds -- is redrawn: out of contract.)
fn draw_scalar<R: Rng + ?Sized>(rng: &mut R) -> u64 {
    loop {
        let mut b = [0u8; 8];
        rng.fill(&mut b);
        let v = i64::from_be_bytes(b);
        if v != 0 && v != i64::MIN {
            return v.unsigned_abs();
        }
    }
}

fn keys_wire<'a>(keys: impl Iterator<Item = &'a PublicKey>) -> Vec<u8> {
    let mut out = Vec::new();
    for k in keys {
        out.extend_from_slice(&g1_wire(&k.point));
    }
    out
}

impl AggregatePublicKey {
    /// aggregates.rs:29-39
    pub fn aggregate(keys: &[&PublicKey]) -> Result<Self, AmclError> {
        Self::sum(keys_wire(keys.iter().copied()), keys.len())
    }
    /// aggregates.rs:46-56
    pub fn into_aggregate(keys: &[PublicKey]) -> Result<Self, AmclError> {
        Self::sum(keys_wire(keys.iter()), keys.len())
    }
    fn sum(pks: Vec<u8>, n: usize) -> Result<Self, AmclError> {
        if n == 0 {
            return Err(AmclError::AggregateEmptyPoints);
        }
        let off = [0u32, n as u32];
        let mut out = [0u8; G1_WIRE];
        let mut st = 0i32;
        let rc = with_ctx(|ctx| unsafe { b3_g1_aggregate(ctx, pks.as_ptr(), off.as_ptr(), 1, out.as_mut_ptr(), &mut st) });
        match rc {
            Some(B3_OK) if st == 0 => Ok(Self { point: g1_from_wire(&out)? }),
            Some(B3_OK) => Err(amcl_error(st)),
            _ => Err(AmclError::InvalidPoint),
        }
    }
}

impl AggregateSignature {
    /// aggregates.rs:100-106
    pub fn aggregate(signatures: &[&Signature]) -> Self {
        if signatures.is_empty() {
            return AggregateSignature::new();
        }
        let mut sigs = Vec::with_capacity(G2_WIRE * signatures.len());
        for s in signatures {
            sigs.extend_from_slice(&g2_wire(&s.point));
        }
        let off = [0u32, signatures.len() as u32];
        let mut out = [0u8; G2_WIRE];
        let mut st = 0i32;
        let rc = with_ctx(|ctx| unsafe { b3_g2_aggregate(ctx, sigs.as_ptr(), off.as_ptr(), 1, out.as_mut_ptr(), &mut st) });
        match (rc, g2_from_wire(&out)) {
            (Some(B3_OK), Ok(point)) if st == 0 => AggregateSignature { point },
            _ => AggregateSignature::new(),
        }
    }

    /// aggregates.rs:130-170
    pub fn aggregate_verify(&self, msgs: &[&[u8]], public_keys: &[&PublicKey]) -> bool {
        if msgs.len() != public_keys.len() || msgs.is_empty() {
            return false;
        }
        let sig = g2_wire(&self.point);
        let pks = keys_wire(public_keys.iter().copied());
        let (blob, off) = pack(msgs.iter().copied());
        let mut accept = 0i32;
        let rc = with_ctx(|ctx| unsafe {
            b3_aggregate_verify(ctx, sig.as_ptr(), pks.as_ptr(), blob.as_ptr(), off.as_ptr(), msgs.len(), &mut accept, std::ptr::null_mut())
        });
        rc == Some(B3_OK) && accept == 1
    }

    /// aggregates.rs:177-215
    pub fn fast_aggregate_verify(&self, msg: &[u8], public_keys: &[&PublicKey]) -> bool {
        if public_keys.is_empty() {
            return false;
        }
        let sig = g2_wire(&self.point);
        let pks = keys_wire(public_keys.iter().copied());
        let mut accept = 0i32;
        let rc = with_ctx(|ctx| unsafe {
            b3_fast_aggregate_verify(ctx, sig.as_ptr(), pks.as_ptr(), public_keys.len(), msg.as_ptr(), msg.len(), &mut accept, std::ptr::null_mut())
        });
        rc == Some(B3_OK) && accept == 1
    }

    /// aggregates.rs:223-253
    pub fn fast_aggregate_verify_pre_aggregated(&self, msg: &[u8], aggregate_public_key: &AggregatePublicKey) -> bool {
        let (sig, apk) = (g2_wire(&self.point), g1_wire(&aggregate_public_key.point));
        let mut accept = 0i32;
        let rc = with_ctx(|ctx| unsafe {
            b3_fast_aggregate_verify_pre_aggregated(ctx, sig.as_ptr(), apk.as_ptr(), msg.as_ptr(), msg.len(), &mut accept, std::ptr::null_mut())
        });
        rc == Some(B3_OK) && accept == 1
    }

    /// aggregates.rs:261-316.  TWO PHASES, so that the caller's RNG is consumed exactly as the reference consumes it
    /// (aggregates.rs:272-287: the scalar of set j is drawn only after signatures 0..=j passed subgroup_check_g2, and
    /// nothing is drawn for or after the first failing set) without any work done twice:
    ///   1. b3_sig_precheck: upload, parse and subgroup-check all signatures -> first_bad;
    ///   2. draw min(first_bad, n) scalars; if every signature passed, b3_verify_multiple_checked runs the batch equation on
    ///      the signatures left in the context by phase 1.
    pub fn verify_multiple_aggregate_signatures<'a, R, I>(rng: &mut R, signature_sets: I) -> bool
    where
        R: Rng + ?Sized,
        I: Iterator<Item = (&'a AggregateSignature, &'a AggregatePublicKey, &'a [u8])>,
    {
        let (mut sigs, mut apks, mut msgs) = (Vec::new(), Vec::new(), Vec::new());
        let mut off = vec![0u32];
        for (s, k, m) in signature_sets {
            sigs.extend_from_slice(&g2_wire(&s.point));
            apks.extend_from_slice(&g1_wire(&k.point));
            msgs.extend_from_slice(m);
            off.push(msgs.len() as u32);
        }
        let n = off.len() - 1;
        if n == 0 {
            return true; // aggregates.rs:266-316 on an empty iterator: the product is empty, e(O, -G1) == 1
        }
        with_ctx(|ctx| {
            let mut first_bad = -1i64;
            if unsafe { b3_sig_precheck(ctx, sigs.as_ptr(), n, &mut first_bad) } != B3_OK {
                return false;
            }
            let n_draw = if first_bad >= 0 { first_bad as usize } else { n };
            let scalars: Vec<u64> = (0..n_draw).map(|_| draw_scalar(rng)).collect();
            if first_bad >= 0 {
                return false;
            }
            let mut accept = 0i32;
            let rc = unsafe {
                b3_verify_multiple_checked(ctx, apks.as_ptr(), std::ptr::null(), msgs.as_ptr(), off.as_ptr(), scalars.as_ptr(), n, &mut accept,
                                           std::ptr::null_mut())
            };
            rc == B3_OK && accept == 1
        })
        .unwrap_or(false)
    }

    /// The same over a device-resident key table (not in the reference: the form a client with a fixed validator set uses).
    /// Set j = (signature, indices of its public keys in `table`, message): the keys are aggregated on the device from decoded
    /// table entries, so 4 bytes per key cross PCIe instead of 96 and nothing is parsed or re-validated per call.
    pub fn verify_multiple_indexed<'a, R, I>(rng: &mut R, table: &KeyTable, signature_sets: I) -> bool
    where
        R: Rng + ?Sized,
        I: Iterator<Item = (&'a AggregateSignature, &'a [u32], &'a [u8])>,
    {
        let (mut sigs, mut idx, mut msgs) = (Vec::new(), Vec::new(), Vec::new());
        let (mut koff, mut moff) = (vec![0u32], vec![0u32]);
        for (s, k, m) in signature_sets {
            sigs.extend_from_slice(&g2_wire(&s.point));
            idx.extend_from_slice(k);
            koff.push(idx.len() as u32);
            msgs.extend_from_slice(m);
            moff.push(msgs.len() as u32);
        }
        let n = moff.len() - 1;
        if n == 0 {
            return true;
        }
        with_ctx(|ctx| {
            let mut first_bad = -1i64;
            if unsafe { b3_sig_precheck(ctx, sigs.as_ptr(), n, &mut first_bad) } != B3_OK {
                return false;
            }
            let n_draw = if first_bad >= 0 { first_bad as usize } else { n };
            let scalars: Vec<u64> = (0..n_draw).map(|_| draw_scalar(rng)).collect();
            if first_bad >= 0 {
                return false;
            }
            let (mut accept, mut fb) = (0i32, -1i64);
            let rc = unsafe {
                b3_verify_multiple_indexed(ctx, table.0, std::ptr::null(), idx.as_ptr(), koff.as_ptr(), msgs.as_ptr(), moff.as_ptr(),
                                           scalars.as_ptr(), n, &mut accept, &mut fb, std::ptr::null_mut())
            };
            rc == B3_OK && accept == 1
        })
        .unwrap_or(false)
    }

    /// Extension (not in the reference): verify_multiple_aggregate_signatures with every DISTINCT message hashed and paired
    /// once (b3_verify_multiple_grouped), for batches whose sets repeat messages -- sync-committee messages, the unaggregated
    /// attestations of one committee.  Messages are deduplicated by their bytes.  The result and the RNG consumption are those
    /// of verify_multiple_aggregate_signatures: b3_sig_precheck -> draw -> the grouped call.
    pub fn verify_multiple_aggregate_signatures_grouped<'a, R, I>(rng: &mut R, signature_sets: I) -> bool
    where
        R: Rng + ?Sized,
        I: Iterator<Item = (&'a AggregateSignature, &'a AggregatePublicKey, &'a [u8])>,
    {
        let (mut sigs, mut apks, mut msgs) = (Vec::new(), Vec::new(), Vec::new());
        let (mut off, mut idx) = (vec![0u32], Vec::new());
        let mut seen: std::collections::HashMap<&'a [u8], u32> = std::collections::HashMap::new();
        for (s, k, m) in signature_sets {
            sigs.extend_from_slice(&g2_wire(&s.point));
            apks.extend_from_slice(&g1_wire(&k.point));
            let next = seen.len() as u32;
            let id = *seen.entry(m).or_insert_with(|| {
                msgs.extend_from_slice(m);
                off.push(msgs.len() as u32);
                next
            });
            idx.push(id);
        }
        let n = idx.len();
        if n == 0 {
            return true;
        }
        with_ctx(|ctx| {
            let mut first_bad = -1i64;
            if unsafe { b3_sig_precheck(ctx, sigs.as_ptr(), n, &mut first_bad) } != B3_OK {
                return false;
            }
            let n_draw = if first_bad >= 0 { first_bad as usize } else { n };
            let scalars: Vec<u64> = (0..n_draw).map(|_| draw_scalar(rng)).collect();
            if first_bad >= 0 {
                return false;
            }
            let (mut accept, mut fb) = (0i32, -1i64);
            let rc = unsafe {
                b3_verify_multiple_grouped(ctx, std::ptr::null(), std::ptr::null(), apks.as_ptr() as *const std::os::raw::c_void,
                                           std::ptr::null(), msgs.as_ptr(), off.as_ptr(), off.len() - 1, idx.as_ptr(), scalars.as_ptr(), n, 0,
                                           &mut accept, &mut fb, std::ptr::null_mut())
            };
            rc == B3_OK && accept == 1
        })
        .unwrap_or(false)
    }

    /// Extension (not in the reference): one verdict per set, `true` where the set ALONE passes
    /// verify_multiple_aggregate_signatures -- what a caller needs after a batch returned false, to attribute and drop the bad
    /// sets.  Exactly one scalar is drawn per set, in order, for every set (no stop at the first bad set: every set gets a
    /// verdict).  One b3_verify_multiple call; if it rejects, b3_verify_multiple_locate reads the per-set verdicts from what
    /// that call left on the device.  A malformed point (or any other failure) gives all `false`.
    pub fn verify_multiple_aggregate_signatures_per_set<'a, R, I>(rng: &mut R, signature_sets: I) -> Vec<bool>
    where
        R: Rng + ?Sized,
        I: Iterator<Item = (&'a AggregateSignature, &'a AggregatePublicKey, &'a [u8])>,
    {
        let (mut sigs, mut apks, mut msgs) = (Vec::new(), Vec::new(), Vec::new());
        let mut off = vec![0u32];
        for (s, k, m) in signature_sets {
            sigs.extend_from_slice(&g2_wire(&s.point));
            apks.extend_from_slice(&g1_wire(&k.point));
            msgs.extend_from_slice(m);
            off.push(msgs.len() as u32);
        }
        let n = off.len() - 1;
        let scalars: Vec<u64> = (0..n).map(|_| draw_scalar(rng)).collect();
        if n == 0 {
            return Vec::new();
        }
        with_ctx(|ctx| {
            let (mut accept, mut fb) = (0i32, -1i64);
            let rc = unsafe {
                b3_verify_multiple(ctx, sigs.as_ptr(), apks.as_ptr(), std::ptr::null(), msgs.as_ptr(), off.as_ptr(), scalars.as_ptr(), n,
                                   &mut accept, &mut fb, std::ptr::null_mut())
            };
            if rc != B3_OK {
                return vec![false; n];
            }
            if accept == 1 {
                return vec![true; n];
            }
            let mut valid = vec![0i32; n];
            if unsafe { b3_verify_multiple_locate(ctx, n, valid.as_mut_ptr(), std::ptr::null_mut()) } != B3_OK {
                return vec![false; n];
            }
            valid.iter().map(|&v| v != 0).collect()
        })
        .unwrap_or_else(|| vec![false; n])
    }

    /// aggregates.rs:319-322
    pub fn from_bytes(bytes: &[u8]) -> Result<AggregateSignature, AmclError> {
        Ok(AggregateSignature { point: Signature::from_bytes(bytes)?.point })
    }
    /// aggregates.rs:325-327
    pub fn as_bytes(&self) -> [u8; G2_BYTES] {
        Signature { point: self.point.clone() }.as_bytes()
    }
}

fn pack<'a>(msgs: impl Iterator<Item = &'a [u8]>) -> (Vec<u8>, Vec<u32>) {
    let (mut blob, mut off) = (Vec::new(), vec![0u32]);
    for m in msgs {
        blob.extend_from_slice(m);
        off.push(blob.len() as u32);
    }
    (blob, off)
}
