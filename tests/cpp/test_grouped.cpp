// C++ host-side test of the grouped extension AggregateSignature::verify_multiple_aggregate_signatures_grouped
// (include/milagro_bls_b200.hpp): every distinct message hashed and paired once (b3_verify_multiple_grouped), with the result
// and the RNG consumption of verify_multiple_aggregate_signatures, for repeated and unique messages, and the grouped C entry's
// locate and argument rules underneath.  Signatures are synthesised with the library's input helpers (pk = [sk]G1,
// sig = [sk]H(msg)).  Needs an sm_100 device; exit code 0 = all checks passed.
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/milagro_bls_b200.hpp"

using namespace milagro_bls;

static int failures = 0;
#define CHECK(cond)                                                                     \
    do {                                                                                \
        if (!(cond)) { std::printf("FAIL %s:%d  %s\n", __FILE__, __LINE__, #cond); failures++; } \
    } while (0)

// deterministic byte stream standing in for rand::Rng (SplitMix64), counting what the callee consumes
struct CountingRng {
    uint64_t x;
    size_t consumed = 0;
    explicit CountingRng(uint64_t seed) : x(seed) {}
    uint64_t next() {
        x += 0x9E3779B97F4A7C15ull;
        uint64_t z = x;
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        return z ^ (z >> 31);
    }
    void fill_bytes(uint8_t* p, size_t n) {
        consumed += n;
        for (size_t i = 0; i < n; i++) p[i] = static_cast<uint8_t>(next());
    }
};

struct Keypair {
    uint8_t sk[32];
    PublicKey pk;
};
static Keypair keypair(uint64_t k) {
    Keypair kp{};
    for (int i = 0; i < 8; i++) kp.sk[31 - i] = static_cast<uint8_t>(k >> (8 * i));
    b3_g1_mul_gen(detail::ctx(), kp.sk, 1, kp.pk.point.data());
    return kp;
}
static Signature sign(const Keypair& kp, const std::string& msg) {           // sig = [sk] hash_to_curve_g2(msg)
    const uint32_t off[2] = {0, static_cast<uint32_t>(msg.size())};
    uint8_t h[192];
    Signature s;
    b3_hash_to_g2(detail::ctx(), reinterpret_cast<const uint8_t*>(msg.data()), off, 1, nullptr, 0, h);
    b3_g2_mul(detail::ctx(), h, kp.sk, 1, s.point.data());
    return s;
}
static const uint8_t* bytes(const std::string& s) { return reinterpret_cast<const uint8_t*>(s.data()); }

int main() {
    if (!detail::ctx()) { std::printf("no sm_100 device / library: the product has no CPU path\n"); return 2; }
    const int n = 8;
    const std::string pool[3] = {"grouped slot root", "grouped attestation data", "grouped other"};
    std::vector<std::string> msgs;
    std::vector<AggregateSignature> sigs(n);
    std::vector<AggregatePublicKey> apks(n);
    for (int j = 0; j < n; j++) {
        Keypair k1 = keypair(7000 + 13 * j), k2 = keypair(9000 + 29 * j);
        msgs.push_back(pool[j % 3 == 2 ? 2 : j % 2]);                        // three messages, repeated
        Signature s1 = sign(k1, msgs[j]), s2 = sign(k2, msgs[j]);
        sigs[j] = AggregateSignature::aggregate({&s1, &s2});
        apks[j] = AggregatePublicKey::into_aggregate({k1.pk, k2.pk}).value;
    }
    auto sets_of = [&](const std::vector<AggregateSignature>& sg, const std::vector<std::string>& ms) {
        std::vector<AggregateSignature::Set> v;
        for (int j = 0; j < n; j++) v.push_back({&sg[j], &apks[j], bytes(ms[j]), ms[j].size()});
        return v;
    };
    std::vector<std::string> unique = msgs;
    for (int j = 0; j < n; j++) unique[j] += " #" + std::to_string(j);
    std::vector<AggregateSignature> usigs = sigs;
    std::vector<AggregatePublicKey> uapks = apks;
    {   // repeated messages, all valid: accepted, one draw per set -- as the ungrouped function
        CountingRng rng(1), ref(1);
        auto sets = sets_of(sigs, msgs);
        CHECK(AggregateSignature::verify_multiple_aggregate_signatures_grouped(rng, sets.begin(), sets.end()));
        CHECK(AggregateSignature::verify_multiple_aggregate_signatures(ref, sets.begin(), sets.end()));
        CHECK(rng.consumed == n * 8 && ref.consumed == rng.consumed);
        int32_t valid[n];
        CHECK(b3_verify_multiple_locate(detail::ctx(), n, valid, nullptr) == B3_OK);     // the ungrouped call enabled it
    }
    {   // a signature of another message (set 3 carries set 2's): rejected by both, same draws
        CountingRng rng(2), ref(2);
        std::vector<AggregateSignature> swapped = sigs;
        swapped[3] = sigs[2];
        auto sets = sets_of(swapped, msgs);
        CHECK(!AggregateSignature::verify_multiple_aggregate_signatures_grouped(rng, sets.begin(), sets.end()));
        int32_t valid[n];
        size_t n_bad = 0;
        CHECK(b3_verify_multiple_locate(detail::ctx(), n, valid, &n_bad) == B3_OK && n_bad == 1 && valid[3] == 0);   // locate after grouped
        CHECK(!AggregateSignature::verify_multiple_aggregate_signatures(ref, sets.begin(), sets.end()));
        CHECK(rng.consumed == n * 8 && ref.consumed == rng.consumed);
    }
    {   // a malformed signature (set 5): the precheck fails before any draw, in both
        CountingRng rng(3), ref(3);
        std::vector<AggregateSignature> bad = sigs;
        bad[5].point[0] ^= 0x01;                                             // off the curve: the precheck fails, nothing is drawn
        auto sets = sets_of(bad, msgs);
        CHECK(!AggregateSignature::verify_multiple_aggregate_signatures_grouped(rng, sets.begin(), sets.end()));
        CHECK(!AggregateSignature::verify_multiple_aggregate_signatures(ref, sets.begin(), sets.end()));
        CHECK(rng.consumed == ref.consumed);
    }
    {   // unique messages (nothing shared)
        CountingRng rng(4), ref(4);
        auto sets = sets_of(sigs, unique);                                   // signatures of the pool messages: all invalid
        CHECK(!AggregateSignature::verify_multiple_aggregate_signatures_grouped(rng, sets.begin(), sets.end()));
        CHECK(!AggregateSignature::verify_multiple_aggregate_signatures(ref, sets.begin(), sets.end()));
        CHECK(rng.consumed == n * 8 && ref.consumed == rng.consumed);
        for (int j = 0; j < n; j++) {
            Keypair k1 = keypair(7000 + 13 * j), k2 = keypair(9000 + 29 * j);
            Signature s1 = sign(k1, unique[j]), s2 = sign(k2, unique[j]);
            usigs[j] = AggregateSignature::aggregate({&s1, &s2});
        }
        auto good = sets_of(usigs, unique);
        CountingRng rng2(5);
        CHECK(AggregateSignature::verify_multiple_aggregate_signatures_grouped(rng2, good.begin(), good.end()));
        CHECK(rng2.consumed == n * 8);
    }
    {   // the C entry's argument rules: n_msgs == 0 and an out-of-range index are refused, the next call is unaffected
        std::vector<uint8_t> sg, ap, blob;
        std::vector<uint32_t> off{0};
        for (int j = 0; j < n; j++) {
            sg.insert(sg.end(), sigs[j].point.begin(), sigs[j].point.end());
            ap.insert(ap.end(), apks[j].point.begin(), apks[j].point.end());
        }
        for (const std::string& m : pool) { blob.insert(blob.end(), m.begin(), m.end()); off.push_back(static_cast<uint32_t>(blob.size())); }
        std::vector<uint32_t> idx(n);
        for (int j = 0; j < n; j++) idx[j] = j % 3 == 2 ? 2 : j % 2;
        std::vector<uint64_t> sc(n);
        for (int j = 0; j < n; j++) sc[j] = 0x1234567ull * (j + 1);
        int accept = -1;
        int64_t fb = 0;
        CHECK(b3_verify_multiple_grouped(detail::ctx(), nullptr, sg.data(), ap.data(), nullptr, blob.data(), off.data(), 0, idx.data(), sc.data(), n, 0,
                                         &accept, &fb, nullptr) == B3_ERR_ARG);
        std::vector<uint32_t> bad_idx = idx;
        bad_idx[6] = 3;
        CHECK(b3_verify_multiple_grouped(detail::ctx(), nullptr, sg.data(), ap.data(), nullptr, blob.data(), off.data(), 3, bad_idx.data(), sc.data(), n,
                                         0, &accept, &fb, nullptr) == B3_ERR_ARG);
        int32_t valid[n];
        CHECK(b3_verify_multiple_locate(detail::ctx(), n, valid, nullptr) == B3_ERR_ARG);
        CHECK(b3_verify_multiple_grouped(detail::ctx(), nullptr, sg.data(), ap.data(), nullptr, blob.data(), off.data(), 3, idx.data(), sc.data(), n, 0,
                                         &accept, &fb, nullptr) == B3_OK && accept == 1 && fb == -1);
        CHECK(b3_verify_multiple_locate(detail::ctx(), n, valid, nullptr) == B3_OK);
        accept = 0;
        CHECK(b3_verify_multiple_grouped(detail::ctx(), nullptr, sg.data(), ap.data(), nullptr, blob.data(), off.data(), 3, idx.data(), sc.data(), 0, 0,
                                         &accept, &fb, nullptr) == B3_OK && accept == 1);
    }
    {   // empty batch: true, nothing drawn
        CountingRng rng(6);
        std::vector<AggregateSignature::Set> none;
        CHECK(AggregateSignature::verify_multiple_aggregate_signatures_grouped(rng, none.begin(), none.end()));
        CHECK(rng.consumed == 0);
    }
    if (failures) std::printf("%d check(s) FAILED\n", failures);
    else std::printf("all checks passed\n");
    return failures ? 1 : 0;
}
