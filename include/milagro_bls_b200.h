/* milagro_bls_b200 -- C ABI of the B200-native BLS12-381 batch-verification engine.
 *
 * Drop-in boundary for the VERIFICATION path of sigp/milagro_bls.  The reference has no FFI: its boundary is
 * the Rust public API (M/src/lib.rs:17-22, M = /root/reference/src).  Each entry point below names the Rust
 * item it replaces; a thin Rust shim (INTEGRATION.md) keeps the reference's signatures and calls these.
 *
 * Wire formats (exactly what the reference's own (de)serialisers produce, A = amcl src dir):
 *   G1 uncompressed  96 B : x || y, 48-byte big-endian each; infinity = 0x40 then zeros   (A/bls381/core.rs:177-190)
 *   G2 uncompressed 192 B : x.im || x.re || y.im || y.re;     infinity = 0x40 then zeros   (A/bls381/core.rs:344-364)
 *   G1 compressed    48 B, G2 compressed 96 B : ZCash flags C/I/S in the top three bits    (A/bls381/core.rs:145-172,312-339)
 *   GT              576 B : 12 x 48-byte big-endian, order of FP12::to_bytes                (A/fp12.rs:859-913)
 *   scalars               : uint64, drawn by the caller with the rule of M/src/aggregates.rs:278-287
 *
 * All pointers are HOST memory unless the name ends in _dev.  Every call is synchronous on the context's
 * stream.  A context is bound to one CUDA device and must not be used from two threads at once; create one
 * context per thread (the reference types are Send+Sync and re-entrant; so is this API across contexts).
 *
 * There is no CPU fallback: every function returns B3_ERR_CUDA if no usable sm_100 device is present.
 */
#ifndef MILAGRO_BLS_B200_H
#define MILAGRO_BLS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* error codes: 0 = ok; -1..-8 mirror AmclError (A/errors.rs:1-11) in declaration order */
#define B3_OK 0
#define B3_ERR_AGGREGATE_EMPTY_POINTS (-1)
#define B3_ERR_HASH_TO_FIELD (-2)
#define B3_ERR_INVALID_SECRET_KEY_SIZE (-3)
#define B3_ERR_INVALID_SECRET_KEY_RANGE (-4)
#define B3_ERR_INVALID_POINT (-5)
#define B3_ERR_INVALID_G1_SIZE (-6)
#define B3_ERR_INVALID_G2_SIZE (-7)
#define B3_ERR_INVALID_YFLAG (-8)
#define B3_ERR_CUDA (-100)
#define B3_ERR_ARG (-101)

typedef struct b3_ctx b3_ctx;

int b3_ctx_create(int device, b3_ctx** out);
void b3_ctx_destroy(b3_ctx* ctx);
const char* b3_last_error(b3_ctx* ctx);
/* cudaStream_t of the context (as void*), so callers can order their own device work against it */
void* b3_ctx_stream(b3_ctx* ctx);
/* number of kernel launches issued by this context so far (bench.py reports it as gpu_launches) */
uint64_t b3_ctx_launch_count(b3_ctx* ctx);
/* device time in ms of the most recent call's kernels, and of its dominant (Miller-loop) kernel */
float b3_ctx_last_kernel_ms(b3_ctx* ctx, int which);
/* per-stage device time (ms, CUDA events on the context's stream) of the most recent verification / hash call;
 * stages 0 .. b3_stage_count()-1 are named by b3_stage_name() */
float b3_ctx_stage_ms(b3_ctx* ctx, int stage);
const char* b3_stage_name(int stage);
/* serial != 0: run the independent stages of a verification call one after another on the context's stream (for
 * per-stage timing); default 0: they overlap on internal streams, joined before the Miller loop */
void b3_ctx_set_serial(b3_ctx* ctx, int serial);
/* finishing kernel of b3_verify_batch: 0 = chosen by batch size (default), 1 = one CTA per item, 3 = one lane pair per item */
void b3_ctx_set_item_kernel(b3_ctx* ctx, int which);
/* The aggregation kernels check that every key / signature they add is ON THE CURVE (the reference's types cannot hold any
 * other point: every constructor checks, M/src/keys.rs:140-175, M/src/signature.rs:43-46).  trusted != 0 declares that the
 * point arrays passed to this context come out of this library's own decompress / validate / aggregate calls (the
 * reference's type invariant) and skips that check.  Default 0. */
void b3_ctx_set_trusted_points(b3_ctx* ctx, int trusted);
/* Chain kernels of a verify_multiple call (subgroup checks, [c]apk, Miller point chains): 0 (default) = the replicated-lane
 * form -- twice the lanes per item, lower latency, ~25 % more arithmetic -- when the call is the only one in flight on its
 * device and has at most 16384 sets, the plain form otherwise; 1 = always replicated; 2 = always plain. */
void b3_ctx_set_latency_mode(b3_ctx* ctx, int mode);
int b3_stage_count(void);

/* ---- (de)serialisation: PublicKey::{from_bytes, from_bytes_unchecked, as_bytes} (M/src/keys.rs:140-160),
 *      Signature::{from_bytes, as_bytes} (M/src/signature.rs:43-51), AggregateSignature::{from_bytes, as_bytes}
 *      (M/src/aggregates.rs:319-327), decompress_g1/g2 + compress_g1/g2 (M/src/amcl_utils.rs:46-74).
 *      status[i] = B3_OK or the AmclError code of item i; the call itself fails only on CUDA/argument errors. */
int b3_g1_decompress(b3_ctx*, const uint8_t* in48, size_t n, int validate /* key_validate, keys.rs:181-186 */,
                     uint8_t* out96, int32_t* status);
int b3_g2_decompress(b3_ctx*, const uint8_t* in96, size_t n, uint8_t* out192, int32_t* status);
int b3_g1_compress(b3_ctx*, const uint8_t* in96, size_t n, uint8_t* out48, int32_t* status);
int b3_g2_compress(b3_ctx*, const uint8_t* in192, size_t n, uint8_t* out96, int32_t* status);
/* PublicKey::from_uncompressed_bytes / key_validate (M/src/keys.rs:163-186): status[i] = B3_OK iff on curve;
 * valid[i] = 1 iff additionally not infinity and in G1 */
int b3_g1_validate(b3_ctx*, const uint8_t* in96, size_t n, int32_t* status, int32_t* valid);
/* subgroup_check_g2 (A/bls381/core.rs:123-127) on parsed signatures; status as above, ok[i] in {0,1} */
int b3_g2_subgroup_check(b3_ctx*, const uint8_t* in192, size_t n, int32_t* status, int32_t* ok);

/* ---- aggregation: AggregatePublicKey::{aggregate, into_aggregate} (M/src/aggregates.rs:29-56) and
 *      AggregateSignature::aggregate (M/src/aggregates.rs:100-106).  Set s owns points off[s] .. off[s+1]-1.
 *      An empty set yields status[s] = B3_ERR_AGGREGATE_EMPTY_POINTS for G1 (the reference's Err) and infinity for G2. */
int b3_g1_aggregate(b3_ctx*, const uint8_t* pks96, const uint32_t* off, size_t n_sets, uint8_t* out96, int32_t* status);
int b3_g2_aggregate(b3_ctx*, const uint8_t* sigs192, const uint32_t* off, size_t n_sets, uint8_t* out192, int32_t* status);

/* ---- hash_to_curve_g2 (M/src/amcl_utils.rs:33-35 -> A/bls381/core.rs:831-839).  Message i is
 *      msgs[off[i] .. off[i+1]).  dst == NULL selects DST_G2 (A/bls381/proof_of_possession.rs:38).  Any other DST may hold
 *      0 to 255 bytes; a longer one returns B3_ERR_HASH_TO_FIELD and hashes nothing (milagro_bls never passes one). */
int b3_hash_to_g2(b3_ctx*, const uint8_t* msgs, const uint32_t* off, size_t n, const uint8_t* dst, size_t dst_len,
                  uint8_t* out192);

/* ---- verification.  accept mirrors the reference's bool; gt (nullable) receives the 576-byte value the
 *      reference compares with one (FP12 after fexp). ---- */
/* Signature::verify (M/src/signature.rs:27-40) */
int b3_verify(b3_ctx*, const uint8_t sig192[192], const uint8_t pk96[96], const uint8_t* msg, size_t msg_len,
              int* accept, uint8_t* gt576);
/* AggregateSignature::fast_aggregate_verify (M/src/aggregates.rs:177-215); n_pks == 0 -> accept = 0 */
int b3_fast_aggregate_verify(b3_ctx*, const uint8_t sig192[192], const uint8_t* pks96, size_t n_pks,
                             const uint8_t* msg, size_t msg_len, int* accept, uint8_t* gt576);
/* AggregateSignature::fast_aggregate_verify_pre_aggregated (M/src/aggregates.rs:223-253) */
int b3_fast_aggregate_verify_pre_aggregated(b3_ctx*, const uint8_t sig192[192], const uint8_t apk96[96],
                                            const uint8_t* msg, size_t msg_len, int* accept, uint8_t* gt576);
/* AggregateSignature::aggregate_verify (M/src/aggregates.rs:130-170); n == 0 -> accept = 0 */
int b3_aggregate_verify(b3_ctx*, const uint8_t sig192[192], const uint8_t* pks96, const uint8_t* msgs,
                        const uint32_t* msg_off, size_t n, int* accept, uint8_t* gt576);
/* AggregateSignature::verify_multiple_aggregate_signatures (M/src/aggregates.rs:261-316).
 * Set j = (sigs192[j], apk_j, msg_j, scalars[j]).  apk_j is either apks96[j] (pk_off == NULL) or the sum of
 * pks96[pk_off[j] .. pk_off[j+1]) aggregated on the device (the C4/C5 shape: 128 keys per set).
 * first_bad (nullable) = index of the first signature failing subgroup_check_g2, or -1; if it is >= 0,
 * accept = 0 exactly as the reference returns false at that set.  n == 0 -> accept = 1. */
int b3_verify_multiple(b3_ctx*, const uint8_t* sigs192, const uint8_t* pks96, const uint32_t* pk_off,
                       const uint8_t* msgs, const uint32_t* msg_off, const uint64_t* scalars, size_t n,
                       int* accept, int64_t* first_bad, uint8_t* gt576);

/* The same in two phases, keeping the reference's RNG contract (M/src/aggregates.rs:272-287: the scalar of set j is drawn only
 * after signatures 0..j passed subgroup_check_g2; nothing is drawn for or after the first failing set) without any work done
 * twice.  b3_sig_precheck uploads, parses and subgroup-checks the signatures and returns first_bad (-1: all passed; a malformed
 * signature returns its AmclError code).  The caller draws min(first_bad, n) scalars; if first_bad < 0 it calls
 * b3_verify_multiple_checked (or b3_verify_multiple_indexed with sigs192 == NULL) ON THE SAME CONTEXT with the same n, which
 * reuses the checked signatures.  Any scalar equal to 0 is rejected with B3_ERR_ARG by every verify_multiple entry: the
 * reference's draw rule never yields it, and it would drop its set from the batch equation. */
int b3_sig_precheck(b3_ctx*, const uint8_t* sigs192, size_t n, int64_t* first_bad);
int b3_verify_multiple_checked(b3_ctx*, const uint8_t* pks96, const uint32_t* pk_off, const uint8_t* msgs,
                               const uint32_t* msg_off, const uint64_t* scalars, size_t n, int* accept, uint8_t* gt576);

/* ---- device-resident public-key table (SURVEY.md 8(f)1).  PublicKey::from_bytes -- decompression + key_validate,
 *      M/src/keys.rs:140-147 -- is paid ONCE per validator; verification calls then name keys by u32 index: 4 bytes instead of
 *      96 per key over PCIe, and no parsing, Montgomery conversion or curve check per use.  A table belongs to the device of
 *      the context that created it and is read-only during verification: any number of contexts may share it.
 *      b3_keytable_append: compressed != 0 -> 48-byte ZCash-compressed keys (PublicKey::from_bytes; validate = 0 gives
 *      from_bytes_unchecked), else 96-byte uncompressed (from_uncompressed_bytes, on-curve check always).  status[i]
 *      (nullable) = B3_OK or the AmclError code; a rejected key keeps its slot, marked invalid -- every set naming it fails
 *      with B3_ERR_INVALID_POINT -- so indices stay aligned with the caller's numbering.  first_index (nullable) receives
 *      the index of keys[0].  Not thread-safe against concurrent verification calls when it has to grow. ---- */
typedef struct b3_keytable b3_keytable;
int b3_keytable_create(b3_ctx*, size_t capacity, b3_keytable** out);
void b3_keytable_destroy(b3_keytable*);
size_t b3_keytable_size(const b3_keytable*);
int b3_keytable_append(b3_ctx*, b3_keytable*, const uint8_t* keys, size_t n, int compressed, int validate,
                       int32_t* status, size_t* first_index);
/* entries idx[0..n) back as 96-byte uncompressed keys (PublicKey::as_uncompressed_bytes, M/src/keys.rs:163-165) */
int b3_keytable_get(b3_ctx*, const b3_keytable*, const uint32_t* idx, size_t n, uint8_t* out96, int32_t* status);
/* AggregatePublicKey::into_aggregate (M/src/aggregates.rs:46-56) over table indices: set s = key_idx[off[s] .. off[s+1]) */
int b3_g1_aggregate_indexed(b3_ctx*, const b3_keytable*, const uint32_t* key_idx, const uint32_t* off, size_t n_sets,
                            uint8_t* out96, int32_t* status);
/* b3_verify_multiple with the keys of set j = table entries key_idx[pk_off[j] .. pk_off[j+1]) (pk_off == NULL: one entry per
 * set).  sigs192 == NULL: the signatures of the preceding b3_sig_precheck on this context. */
int b3_verify_multiple_indexed(b3_ctx*, const b3_keytable*, const uint8_t* sigs192, const uint32_t* key_idx,
                               const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off,
                               const uint64_t* scalars, size_t n, int* accept, int64_t* first_bad, uint8_t* gt576);

/* b3_verify_multiple / b3_verify_multiple_indexed on inputs already resident in HBM: every input pointer is DEVICE memory
 * (signature and key records 16-byte aligned); accept, first_bad and gt576 are host pointers. */
int b3_verify_multiple_dev(b3_ctx*, const uint8_t* sigs192_dev, const uint8_t* pks96_dev, const uint32_t* pk_off_dev,
                           const uint8_t* msgs_dev, const uint32_t* msg_off_dev, const uint64_t* scalars_dev, size_t n,
                           int* accept, int64_t* first_bad, uint8_t* gt576);
int b3_verify_multiple_indexed_dev(b3_ctx*, const b3_keytable*, const uint8_t* sigs192_dev, const uint32_t* key_idx_dev,
                                   const uint32_t* pk_off_dev, const uint8_t* msgs_dev, const uint32_t* msg_off_dev,
                                   const uint64_t* scalars_dev, size_t n, int* accept, int64_t* first_bad, uint8_t* gt576);

/* verify_multiple over sets that NAME THEIR MESSAGE BY INDEX (sync-committee messages, unaggregated attestations of one
 * committee, aggregates of one slot): set j = (sigs192[j], the keys of set j as in b3_verify_multiple (table == NULL: 96-byte
 * keys) or b3_verify_multiple_indexed (u32 indices into `table`), message msg_idx[j], scalars[j]); message k is
 * msgs[msg_off[k] .. msg_off[k+1]), k < n_msgs.  Each distinct message is hashed once and gets one Miller pair, whose G1
 * member is the sum of [c_j] apk_j over the sets naming it (prod_j e([c_j] apk_j, H) = e(sum_j [c_j] apk_j, H)); subgroup
 * checks, key aggregation and the scalar multiplications stay per set.  accept, first_bad and gt576 equal, byte for byte,
 * those of b3_verify_multiple / _indexed on the same sets with each set's message written out.  A message no set names, or
 * whose sets' scaled keys sum to infinity, contributes 1.  sigs192 == NULL (host pointers only): the signatures of the
 * preceding b3_sig_precheck.  device_pointers != 0: every input pointer is device memory.  n == 0 -> accept = 1; with n > 0,
 * n_msgs == 0, any msg_idx[j] >= n_msgs or a zero scalar returns B3_ERR_ARG.  b3_verify_multiple_locate works after it. */
int b3_verify_multiple_grouped(b3_ctx*, const b3_keytable* table, const uint8_t* sigs192, const void* keys,
                               const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off, size_t n_msgs,
                               const uint32_t* msg_idx, const uint64_t* scalars, size_t n, int device_pointers, int* accept,
                               int64_t* first_bad, uint8_t* gt576);

/* Per-set verdicts for the most recent WHOLE verify_multiple call on this context (b3_verify_multiple, _checked, _indexed,
 * _dev, _indexed_dev, _grouped) that returned B3_OK.  n must be that call's n.  valid[j] = 1 iff set j ALONE passes
 * verify_multiple_aggregate_signatures (M/src/aggregates.rs:261-316); n_invalid (nullable) = number of zeros.
 * That is: sig_j passed subgroup_check_g2 and e(apk_j, H(msg_j)) == e(sig_j, G1); an aggregate key at infinity (an empty key
 * range, or keys that cancel) contributes 1, so such a set is valid iff sig_j is infinity.  The verdict does not depend on
 * the batch scalars and is computed without randomness.  Locate reuses what the batch call left on the device (hashes to
 * G2 and their Miller lines, aggregate keys, parsed and checked signatures): the new work is one Miller point chain per
 * signature and one two-pair Miller loop + final exponentiation per set.  If that call accepted, every valid[j] = 1 and
 * nothing runs on the device.  Any other call on the context (including b3_sig_precheck, the _partial and sharded entries,
 * b3_verify_batch, b3_hash_to_g2 and b3_keytable_append) ends the window: locate then returns B3_ERR_ARG, as it does for a
 * wrong n.  Locate itself may be repeated and does not change the result of the next call. */
int b3_verify_multiple_locate(b3_ctx*, size_t n, int32_t* valid, size_t* n_invalid);

/* ---- batched verification of n INDEPENDENT items with one accept bit each (SURVEY.md 8(f)3: locating the bad set
 *      after a batch reject, or bulk verification of unrelated signatures).  Item i is, by `mode`,
 *        B3_ITEM_VERIFY          Signature::verify(sig_i, msg_i, pk_i)                           (M/src/signature.rs:27-40)
 *        B3_ITEM_FAST_AGGREGATE  fast_aggregate_verify(sig_i, msg_i, pks96[pk_off[i] .. pk_off[i+1]))  (M/src/aggregates.rs:177-215)
 *        B3_ITEM_PRE_AGGREGATED  fast_aggregate_verify_pre_aggregated(sig_i, msg_i, apk_i)       (M/src/aggregates.rs:223-253)
 *      (pk_off is read only in mode B3_ITEM_FAST_AGGREGATE; otherwise pks96 holds one key per item).
 *      accept[i] = the reference's bool; status[i] = B3_OK or the AmclError code of a malformed input of item i
 *      (B3_ERR_AGGREGATE_EMPTY_POINTS for an empty key list; accept[i] = 0 in every such case);
 *      gt576 (nullable, n x 576 B) = each item's FP12 after fexp, all-zero for items rejected before the pairing.
 *      One final exponentiation PER ITEM: one CTA per item below 2048 items, one lane pair per item above. ---- */
#define B3_ITEM_VERIFY 0
#define B3_ITEM_FAST_AGGREGATE 1
#define B3_ITEM_PRE_AGGREGATED 2
int b3_verify_batch(b3_ctx*, int mode, const uint8_t* sigs192, const uint8_t* pks96, const uint32_t* pk_off,
                    const uint8_t* msgs, const uint32_t* msg_off, size_t n, int32_t* accept, int32_t* status,
                    uint8_t* gt576);

/* ---- device-resident variants (inputs already in HBM; used for multi-GPU sharding and resident benchmarks).
 *      partial_dev receives this rank's Miller-loop product (B3_PARTIAL_BYTES of device memory, internal
 *      Montgomery layout -- only meaningful to b3_combine_partials_dev of the same library build).
 *      The pair (sum_j [c_j] sig_j, -G1) of this rank's sets is already folded into the partial. ---- */
#define B3_PARTIAL_BYTES 592 /* 576 B Fp12 + int64 first_bad + 8 B pad */
int b3_verify_multiple_partial_dev(b3_ctx*, const uint8_t* sigs192_dev, const uint8_t* pks96_dev,
                                   const uint32_t* pk_off_dev, const uint8_t* msgs_dev, const uint32_t* msg_off_dev,
                                   const uint64_t* scalars_dev, size_t n, int64_t index_base, uint8_t* partial_dev);
/* the same with this rank's shard in HOST memory (the sharded form of b3_verify_multiple: M/src/aggregates.rs:261-316 on
 * sets [index_base, index_base + n)); the partial stays on the device for the all-gather */
int b3_verify_multiple_partial(b3_ctx*, const uint8_t* sigs192, const uint8_t* pks96, const uint32_t* pk_off,
                               const uint8_t* msgs, const uint32_t* msg_off, const uint64_t* scalars, size_t n,
                               int64_t index_base, uint8_t* partial_dev);
/* the two partial forms over a key table */
int b3_verify_multiple_indexed_partial(b3_ctx*, const b3_keytable*, const uint8_t* sigs192, const uint32_t* key_idx,
                                       const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off,
                                       const uint64_t* scalars, size_t n, int64_t index_base, uint8_t* partial_dev);
int b3_verify_multiple_indexed_partial_dev(b3_ctx*, const b3_keytable*, const uint8_t* sigs192_dev,
                                           const uint32_t* key_idx_dev, const uint32_t* pk_off_dev, const uint8_t* msgs_dev,
                                           const uint32_t* msg_off_dev, const uint64_t* scalars_dev, size_t n,
                                           int64_t index_base, uint8_t* partial_dev);
/* product of n_partials partials (gathered from all ranks) -> one final exponentiation -> accept, first_bad, gt */
int b3_combine_partials_dev(b3_ctx*, const uint8_t* partials_dev, size_t n_partials, int* accept, int64_t* first_bad,
                            uint8_t* gt576);
int b3_verify_batch_dev(b3_ctx*, int mode, const uint8_t* sigs192_dev, const uint8_t* pks96_dev,
                        const uint32_t* pk_off_dev, const uint8_t* msgs_dev, const uint32_t* msg_off_dev, size_t n,
                        int32_t* accept_dev, int32_t* status_dev, uint8_t* gt576_dev);
int b3_hash_to_g2_dev(b3_ctx*, const uint8_t* msgs_dev, const uint32_t* off_dev, size_t n, uint8_t* out192_dev);
int b3_g1_aggregate_dev(b3_ctx*, const uint8_t* pks96_dev, const uint32_t* off_dev, size_t n_sets, uint8_t* out96_dev,
                        int32_t* status_dev);

/* ---- multi-GPU: the sharded form of verify_multiple_aggregate_signatures (M/src/aggregates.rs:261-316; SURVEY.md 8e).
 *      One process per GPU.  Rank r verifies sets [index_base, index_base + n) of the global batch (scalars drawn for the
 *      GLOBAL set order); the 592-byte partials are combined with ONE ncclAllGather over NVLink / NVSwitch and one final
 *      exponentiation on every rank, so every rank returns the global accept bit, the global first_bad and the GT of the whole
 *      batch.  NCCL is bound at run time (the libnccl.so.2 already in the process, else the system one, or $B3_NCCL_LIB).
 *      b3_nccl_unique_id: call on one rank, ship the 128 bytes to the others by any means (the Rust host's own transport).
 *      A communicator serves `lanes` contexts of this process (one host thread + b3_ctx each); call k of lane t is step k,
 *      and the all-gather of a step carries the partials of all its lanes (issued by the lane that deposits last, on the
 *      communicator's own high-priority stream).  Every rank must use the same `lanes` and make the same calls per lane.
 *      b3_sharded_begin returns once this rank's partial is deposited; b3_sharded_finish combines.  A lane may begin step
 *      k + 1 before finishing step k (at most 3 steps open), which gives the collective a whole call time to complete.
 *      keys = pks96 (table == NULL) or u32 indices into `table`; device_pointers != 0: all input pointers are device memory. ---- */
typedef struct b3_comm b3_comm;
int b3_nccl_unique_id(uint8_t id128[128]);
int b3_comm_create(int device, int nranks, int rank, const uint8_t id128[128], int lanes, b3_comm** out);
void b3_comm_destroy(b3_comm*);
const char* b3_comm_last_error(b3_comm*);
/* number of collectives issued so far (one per step) */
uint64_t b3_comm_collective_count(b3_comm*);
int b3_sharded_begin(b3_ctx*, b3_comm*, int lane, const b3_keytable* table, const uint8_t* sigs192, const void* keys,
                     const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off, const uint64_t* scalars, size_t n,
                     int64_t index_base, int device_pointers, int64_t* ticket);
int b3_sharded_finish(b3_ctx*, b3_comm*, int lane, int64_t ticket, int* accept, int64_t* first_bad, uint8_t* gt576);
int b3_verify_multiple_sharded(b3_ctx*, b3_comm*, int lane, const b3_keytable* table, const uint8_t* sigs192,
                               const void* keys, const uint32_t* pk_off, const uint8_t* msgs, const uint32_t* msg_off,
                               const uint64_t* scalars, size_t n, int64_t index_base, int device_pointers, int* accept,
                               int64_t* first_bad, uint8_t* gt576);

/* ---- signing-side helpers.  OUT of the verification path (the reference's Signature::new / SecretKey live on
 *      the CPU); exported only so tests and bench.py can synthesise valid inputs at full size quickly.
 *      scalars32: n x 32-byte big-endian integers (< 2^256). ---- */
int b3_g1_mul_gen(b3_ctx*, const uint8_t* scalars32, size_t n, uint8_t* out96);
int b3_g2_mul(b3_ctx*, const uint8_t* pts192, const uint8_t* scalars32, size_t n, uint8_t* out192);

/* ---- measurement helper: pure-IMAD roofline microbenchmark (returns 32-bit IMAD lane-ops per second) ---- */
int b3_imad_peak(b3_ctx*, int wide /* 0: IMAD, 1: IMAD.WIDE carry chain */, double* ops_per_s);

#ifdef __cplusplus
}
#endif
#endif
