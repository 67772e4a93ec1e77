// milagro_bls_b200.hpp -- C++17 host mirror of sigp/milagro_bls's verification API over the C ABI of milagro_bls_b200.h.
//
// The reference is compiled code (Rust) whose boundary is its public API (/root/reference/src/lib.rs:17-22); there is no Rust
// toolchain in this image, so this header is the COMPILED-LANGUAGE host side above the C ABI: the same type names, method names,
// argument meaning and error behaviour as the reference, so that tests/cpp/test_api.cpp reads like the reference's own tests.
// (shim/ holds the Rust source a maintainer adds; milagro_bls_b200/api.py is the Python mirror the pytest suite drives.)
//
//   reference (M = /root/reference/src)                      here
//   PublicKey            M/keys.rs:116-186                   milagro_bls::PublicKey
//   Signature            M/signature.rs:9-51                 milagro_bls::Signature           (verification half; no signing)
//   AggregatePublicKey   M/aggregates.rs:17-78               milagro_bls::AggregatePublicKey
//   AggregateSignature   M/aggregates.rs:83-327              milagro_bls::AggregateSignature
//   AmclError            A/errors.rs:1-11                    milagro_bls::AmclError
// Decoding returns Result<T> (the reference's Result<T, AmclError>); every verify* returns a plain bool and maps every failure
// to false; the batch scalars come from a caller-injected RNG (any type with fill_bytes(uint8_t*, size_t)), consumed exactly as
// M/aggregates.rs:272-287 consumes it.  Points are held in the reference's uncompressed wire form (96 / 192 bytes).
// There is no CPU fallback: without the library or an sm_100 device every call fails (verify* -> false, decode -> InvalidPoint).
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <map>
#include <string>
#include <utility>
#include <vector>

#include "milagro_bls_b200.h"

namespace milagro_bls {

constexpr size_t G1_BYTES = 48, G2_BYTES = 96;

enum class AmclError {          // A/errors.rs:1-11, numbered as the B3_ERR_* codes (negated)
    None = 0,
    AggregateEmptyPoints = 1,
    HashToFieldError = 2,
    InvalidSecretKeySize = 3,
    InvalidSecretKeyRange = 4,
    InvalidPoint = 5,
    InvalidG1Size = 6,
    InvalidG2Size = 7,
    InvalidYFlag = 8,
};
inline AmclError amcl_error(int code) { return (code < 0 && code >= -8) ? static_cast<AmclError>(-code) : AmclError::InvalidPoint; }

template <class T>
struct Result {
    T value{};
    AmclError err = AmclError::None;
    bool is_ok() const { return err == AmclError::None; }
    explicit operator bool() const { return is_ok(); }
};

// One verification context per thread (the reference's types are Send + Sync and its functions re-entrant; a b3_ctx is
// single-threaded, contexts are independent).  set_device() applies to contexts created afterwards.
namespace detail {
inline int& device_ref() { static int d = 0; return d; }
struct Holder {
    b3_ctx* ctx = nullptr;
    ~Holder() { if (ctx) b3_ctx_destroy(ctx); }
};
inline b3_ctx* ctx() {
    thread_local Holder h;
    if (!h.ctx && b3_ctx_create(device_ref(), &h.ctx) != B3_OK) h.ctx = nullptr;
    return h.ctx;
}
using G1Wire = std::array<uint8_t, 2 * G1_BYTES>;
using G2Wire = std::array<uint8_t, 2 * G2_BYTES>;
inline G1Wire g1_infinity() { G1Wire w{}; w[0] = 0x40; return w; }
inline G2Wire g2_infinity() { G2Wire w{}; w[0] = 0x40; return w; }
}  // namespace detail
inline void set_device(int device) { detail::device_ref() = device; }

struct PublicKey {
    detail::G1Wire point{};
    // M/keys.rs:140-147: decompression + key_validate
    static Result<PublicKey> from_bytes(const uint8_t* bytes, size_t len) { return decode(bytes, len, 1); }
    // M/keys.rs:150-155
    static Result<PublicKey> from_bytes_unchecked(const uint8_t* bytes, size_t len) { return decode(bytes, len, 0); }
    // M/keys.rs:168-175 (on-curve check only: "MUST only be used on verified keys")
    static Result<PublicKey> from_uncompressed_bytes(const uint8_t* bytes, size_t len) {
        Result<PublicKey> r;
        if (len != 2 * G1_BYTES) { r.err = AmclError::InvalidG1Size; return r; }
        int32_t st = 0, valid = 0;
        b3_ctx* c = detail::ctx();
        if (!c || b3_g1_validate(c, bytes, 1, &st, &valid) != B3_OK) { r.err = AmclError::InvalidPoint; return r; }
        if (st) { r.err = amcl_error(st); return r; }
        std::memcpy(r.value.point.data(), bytes, 2 * G1_BYTES);
        return r;
    }
    // M/keys.rs:158-160
    std::array<uint8_t, G1_BYTES> as_bytes() const {
        std::array<uint8_t, G1_BYTES> out{};
        int32_t st = 0;
        b3_ctx* c = detail::ctx();
        if (c) b3_g1_compress(c, point.data(), 1, out.data(), &st);
        return out;
    }
    // M/keys.rs:163-165
    detail::G1Wire as_uncompressed_bytes() const { return point; }
    // M/keys.rs:181-186: not infinity and in G1
    bool key_validate() const {
        int32_t st = 0, valid = 0;
        b3_ctx* c = detail::ctx();
        return c && b3_g1_validate(c, point.data(), 1, &st, &valid) == B3_OK && st == 0 && valid == 1;
    }
    bool operator==(const PublicKey& o) const { return point == o.point; }

private:
    static Result<PublicKey> decode(const uint8_t* bytes, size_t len, int validate) {
        Result<PublicKey> r;
        if (len != G1_BYTES) { r.err = AmclError::InvalidG1Size; return r; }          // M/amcl_utils.rs:52-58
        int32_t st = 0;
        b3_ctx* c = detail::ctx();
        if (!c || b3_g1_decompress(c, bytes, 1, validate, r.value.point.data(), &st) != B3_OK) { r.err = AmclError::InvalidPoint; return r; }
        if (st) r.err = amcl_error(st);
        return r;
    }
};

struct Signature {
    detail::G2Wire point{};
    // M/signature.rs:27-40
    bool verify(const uint8_t* msg, size_t msg_len, const PublicKey& pk) const {
        int accept = 0;
        b3_ctx* c = detail::ctx();
        return c && b3_verify(c, point.data(), pk.point.data(), msg, msg_len, &accept, nullptr) == B3_OK && accept == 1;
    }
    // M/signature.rs:43-46 (no subgroup check: verify does it)
    static Result<Signature> from_bytes(const uint8_t* bytes, size_t len) {
        Result<Signature> r;
        if (len != G2_BYTES) { r.err = AmclError::InvalidG2Size; return r; }          // M/amcl_utils.rs:68-74
        int32_t st = 0;
        b3_ctx* c = detail::ctx();
        if (!c || b3_g2_decompress(c, bytes, 1, r.value.point.data(), &st) != B3_OK) { r.err = AmclError::InvalidPoint; return r; }
        if (st) r.err = amcl_error(st);
        return r;
    }
    // M/signature.rs:49-51
    std::array<uint8_t, G2_BYTES> as_bytes() const {
        std::array<uint8_t, G2_BYTES> out{};
        int32_t st = 0;
        b3_ctx* c = detail::ctx();
        if (c) b3_g2_compress(c, point.data(), 1, out.data(), &st);
        return out;
    }
    bool operator==(const Signature& o) const { return point == o.point; }
};

struct AggregatePublicKey {
    detail::G1Wire point = detail::g1_infinity();
    // M/aggregates.rs:29-39
    static Result<AggregatePublicKey> aggregate(const std::vector<const PublicKey*>& keys) {
        std::vector<uint8_t> blob;
        blob.reserve(96 * keys.size());
        for (const PublicKey* k : keys) blob.insert(blob.end(), k->point.begin(), k->point.end());
        return sum(blob, keys.size());
    }
    // M/aggregates.rs:46-56
    static Result<AggregatePublicKey> into_aggregate(const std::vector<PublicKey>& keys) {
        std::vector<uint8_t> blob;
        blob.reserve(96 * keys.size());
        for (const PublicKey& k : keys) blob.insert(blob.end(), k.point.begin(), k.point.end());
        return sum(blob, keys.size());
    }
    // M/aggregates.rs:61-63
    static AggregatePublicKey from_public_key(const PublicKey& key) { AggregatePublicKey a; a.point = key.point; return a; }
    // M/aggregates.rs:68-77
    void add(const PublicKey& key) { add_point(key.point); }
    void add_aggregate(const AggregatePublicKey& other) { add_point(other.point); }
    bool operator==(const AggregatePublicKey& o) const { return point == o.point; }

private:
    static Result<AggregatePublicKey> sum(const std::vector<uint8_t>& blob, size_t n) {
        Result<AggregatePublicKey> r;
        if (n == 0) { r.err = AmclError::AggregateEmptyPoints; return r; }
        const uint32_t off[2] = {0, static_cast<uint32_t>(n)};
        int32_t st = 0;
        b3_ctx* c = detail::ctx();
        if (!c || b3_g1_aggregate(c, blob.data(), off, 1, r.value.point.data(), &st) != B3_OK) { r.err = AmclError::InvalidPoint; return r; }
        if (st) r.err = amcl_error(st);
        return r;
    }
    void add_point(const detail::G1Wire& p) {
        uint8_t two[192];
        std::memcpy(two, point.data(), 96);
        std::memcpy(two + 96, p.data(), 96);
        const uint32_t off[2] = {0, 2};
        int32_t st = 0;
        detail::G1Wire out{};
        b3_ctx* c = detail::ctx();
        if (c && b3_g1_aggregate(c, two, off, 1, out.data(), &st) == B3_OK && st == 0) point = out;
    }
};

struct AggregateSignature {
    detail::G2Wire point = detail::g2_infinity();          // AggregateSignature::new: infinity (M/aggregates.rs:93-95)
    // M/aggregates.rs:100-106
    static AggregateSignature aggregate(const std::vector<const Signature*>& signatures) {
        AggregateSignature a;
        if (signatures.empty()) return a;
        std::vector<uint8_t> blob;
        blob.reserve(192 * signatures.size());
        for (const Signature* s : signatures) blob.insert(blob.end(), s->point.begin(), s->point.end());
        const uint32_t off[2] = {0, static_cast<uint32_t>(signatures.size())};
        int32_t st = 0;
        detail::G2Wire out{};
        b3_ctx* c = detail::ctx();
        if (c && b3_g2_aggregate(c, blob.data(), off, 1, out.data(), &st) == B3_OK && st == 0) a.point = out;
        return a;
    }
    // M/aggregates.rs:109-111
    static AggregateSignature from_signature(const Signature& s) { AggregateSignature a; a.point = s.point; return a; }
    // M/aggregates.rs:114-124
    void add(const Signature& s) { add_point(s.point); }
    void add_aggregate(const AggregateSignature& o) { add_point(o.point); }

    // M/aggregates.rs:130-170
    bool aggregate_verify(const std::vector<std::pair<const uint8_t*, size_t>>& msgs, const std::vector<const PublicKey*>& public_keys) const {
        if (msgs.size() != public_keys.size() || msgs.empty()) return false;
        std::vector<uint8_t> pks, blob;
        std::vector<uint32_t> off{0};
        for (const PublicKey* k : public_keys) pks.insert(pks.end(), k->point.begin(), k->point.end());
        for (const auto& m : msgs) { blob.insert(blob.end(), m.first, m.first + m.second); off.push_back(static_cast<uint32_t>(blob.size())); }
        int accept = 0;
        b3_ctx* c = detail::ctx();
        return c && b3_aggregate_verify(c, point.data(), pks.data(), blob.data(), off.data(), msgs.size(), &accept, nullptr) == B3_OK && accept == 1;
    }
    // M/aggregates.rs:177-215
    bool fast_aggregate_verify(const uint8_t* msg, size_t msg_len, const std::vector<const PublicKey*>& public_keys) const {
        if (public_keys.empty()) return false;
        std::vector<uint8_t> pks;
        for (const PublicKey* k : public_keys) pks.insert(pks.end(), k->point.begin(), k->point.end());
        int accept = 0;
        b3_ctx* c = detail::ctx();
        return c && b3_fast_aggregate_verify(c, point.data(), pks.data(), public_keys.size(), msg, msg_len, &accept, nullptr) == B3_OK && accept == 1;
    }
    // M/aggregates.rs:223-253
    bool fast_aggregate_verify_pre_aggregated(const uint8_t* msg, size_t msg_len, const AggregatePublicKey& apk) const {
        int accept = 0;
        b3_ctx* c = detail::ctx();
        return c && b3_fast_aggregate_verify_pre_aggregated(c, point.data(), apk.point.data(), msg, msg_len, &accept, nullptr) == B3_OK && accept == 1;
    }

    // One signature set of verify_multiple_aggregate_signatures: (&AggregateSignature, &AggregatePublicKey, &[u8])
    struct Set {
        const AggregateSignature* signature;
        const AggregatePublicKey* public_key;
        const uint8_t* msg;
        size_t msg_len;
    };
    // M/aggregates.rs:261-316.  Rng: any type with `void fill_bytes(uint8_t*, size_t)` (rand::Rng::fill in the reference).
    // TWO PHASES so that the caller's RNG is consumed exactly as the reference consumes it (M/aggregates.rs:272-287: a set's
    // scalar is drawn only after its signature passed subgroup_check_g2; nothing is drawn for or after the first failing set)
    // without running anything twice: b3_sig_precheck -> draw -> b3_verify_multiple_checked.
    template <class Rng, class It>
    static bool verify_multiple_aggregate_signatures(Rng& rng, It first, It last) {
        std::vector<uint8_t> sigs, apks, msgs;
        std::vector<uint32_t> off{0};
        for (It it = first; it != last; ++it) {
            const Set& s = *it;
            sigs.insert(sigs.end(), s.signature->point.begin(), s.signature->point.end());
            apks.insert(apks.end(), s.public_key->point.begin(), s.public_key->point.end());
            msgs.insert(msgs.end(), s.msg, s.msg + s.msg_len);
            off.push_back(static_cast<uint32_t>(msgs.size()));
        }
        const size_t n = off.size() - 1;
        if (n == 0) return true;
        b3_ctx* c = detail::ctx();
        if (!c) return false;
        int64_t first_bad = -1;
        if (b3_sig_precheck(c, sigs.data(), n, &first_bad) != B3_OK) return false;
        const size_t n_draw = first_bad >= 0 ? static_cast<size_t>(first_bad) : n;
        std::vector<uint64_t> scalars(n_draw);
        for (size_t j = 0; j < n_draw; j++) scalars[j] = draw_scalar(rng);
        if (first_bad >= 0) return false;
        int accept = 0;
        return b3_verify_multiple_checked(c, apks.data(), nullptr, msgs.data(), off.data(), scalars.data(), n, &accept, nullptr) == B3_OK && accept == 1;
    }
    // Extension (not in the reference): verify_multiple_aggregate_signatures with each DISTINCT message hashed and paired once
    // (b3_verify_multiple_grouped), for batches whose sets repeat messages -- sync-committee messages, the unaggregated
    // attestations of one committee.  Messages are deduplicated by their bytes.  The result and the RNG consumption are those
    // of verify_multiple_aggregate_signatures: the same two phases, b3_sig_precheck -> draw -> the grouped call.
    template <class Rng, class It>
    static bool verify_multiple_aggregate_signatures_grouped(Rng& rng, It first, It last) {
        std::vector<uint8_t> sigs, apks, msgs;
        std::vector<uint32_t> off{0}, idx;
        std::map<std::string, uint32_t> seen;
        for (It it = first; it != last; ++it) {
            const Set& s = *it;
            sigs.insert(sigs.end(), s.signature->point.begin(), s.signature->point.end());
            apks.insert(apks.end(), s.public_key->point.begin(), s.public_key->point.end());
            const auto ins = seen.emplace(std::string(reinterpret_cast<const char*>(s.msg), s.msg_len), static_cast<uint32_t>(seen.size()));
            if (ins.second) {
                msgs.insert(msgs.end(), s.msg, s.msg + s.msg_len);
                off.push_back(static_cast<uint32_t>(msgs.size()));
            }
            idx.push_back(ins.first->second);
        }
        const size_t n = idx.size();
        if (n == 0) return true;
        b3_ctx* c = detail::ctx();
        if (!c) return false;
        int64_t first_bad = -1;
        if (b3_sig_precheck(c, sigs.data(), n, &first_bad) != B3_OK) return false;
        const size_t n_draw = first_bad >= 0 ? static_cast<size_t>(first_bad) : n;
        std::vector<uint64_t> scalars(n_draw);
        for (size_t j = 0; j < n_draw; j++) scalars[j] = draw_scalar(rng);
        if (first_bad >= 0) return false;
        int accept = 0;
        return b3_verify_multiple_grouped(c, nullptr, nullptr, apks.data(), nullptr, msgs.data(), off.data(), off.size() - 1, idx.data(),
                                          scalars.data(), n, 0, &accept, nullptr, nullptr) == B3_OK && accept == 1;
    }
    // Extension (not in the reference): one verdict per set, true where the set ALONE passes
    // verify_multiple_aggregate_signatures.  Exactly one scalar is drawn per set, in order, for every set (no stop at the first
    // bad set: every set gets a verdict).  One b3_verify_multiple call; if it rejects, b3_verify_multiple_locate reads the
    // per-set verdicts from what that call left on the device.  A malformed point or any other failure gives all false.
    template <class Rng, class It>
    static std::vector<bool> verify_multiple_aggregate_signatures_per_set(Rng& rng, It first, It last) {
        std::vector<uint8_t> sigs, apks, msgs;
        std::vector<uint32_t> off{0};
        for (It it = first; it != last; ++it) {
            const Set& s = *it;
            sigs.insert(sigs.end(), s.signature->point.begin(), s.signature->point.end());
            apks.insert(apks.end(), s.public_key->point.begin(), s.public_key->point.end());
            msgs.insert(msgs.end(), s.msg, s.msg + s.msg_len);
            off.push_back(static_cast<uint32_t>(msgs.size()));
        }
        const size_t n = off.size() - 1;
        std::vector<uint64_t> scalars(n);
        for (size_t j = 0; j < n; j++) scalars[j] = draw_scalar(rng);
        std::vector<bool> out(n, false);
        if (n == 0) return out;
        b3_ctx* c = detail::ctx();
        int accept = 0;
        if (!c || b3_verify_multiple(c, sigs.data(), apks.data(), nullptr, msgs.data(), off.data(), scalars.data(), n, &accept, nullptr, nullptr) != B3_OK)
            return out;
        if (accept) return std::vector<bool>(n, true);
        std::vector<int32_t> valid(n, 0);
        if (b3_verify_multiple_locate(c, n, valid.data(), nullptr) != B3_OK) return out;
        for (size_t j = 0; j < n; j++) out[j] = valid[j] != 0;
        return out;
    }
    // M/aggregates.rs:278-287: 8 bytes, i64::from_be_bytes(..).abs(), retry while 0 (i64::MIN, whose abs() overflows, is redrawn)
    template <class Rng>
    static uint64_t draw_scalar(Rng& rng) {
        for (;;) {
            uint8_t b[8];
            rng.fill_bytes(b, 8);
            uint64_t v = 0;
            for (int i = 0; i < 8; i++) v = (v << 8) | b[i];
            const int64_t s = static_cast<int64_t>(v);
            if (s == 0 || s == INT64_MIN) continue;
            return static_cast<uint64_t>(s < 0 ? -s : s);
        }
    }

    // M/aggregates.rs:319-327
    static Result<AggregateSignature> from_bytes(const uint8_t* bytes, size_t len) {
        Result<AggregateSignature> r;
        Result<Signature> s = Signature::from_bytes(bytes, len);
        r.err = s.err;
        r.value.point = s.value.point;
        if (!s) r.value.point = detail::g2_infinity();
        return r;
    }
    std::array<uint8_t, G2_BYTES> as_bytes() const { Signature s; s.point = point; return s.as_bytes(); }
    bool operator==(const AggregateSignature& o) const { return point == o.point; }

private:
    void add_point(const detail::G2Wire& p) {
        uint8_t two[384];
        std::memcpy(two, point.data(), 192);
        std::memcpy(two + 192, p.data(), 192);
        const uint32_t off[2] = {0, 2};
        int32_t st = 0;
        detail::G2Wire out{};
        b3_ctx* c = detail::ctx();
        if (c && b3_g2_aggregate(c, two, off, 1, out.data(), &st) == B3_OK && st == 0) point = out;
    }
};

}  // namespace milagro_bls
