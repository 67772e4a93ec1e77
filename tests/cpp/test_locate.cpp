// C++ host-side test of the per-set extension AggregateSignature::verify_multiple_aggregate_signatures_per_set
// (include/milagro_bls_b200.hpp): one verdict per set, true where the set alone passes verify_multiple_aggregate_signatures
// (M/src/aggregates.rs:261-316), one scalar drawn per set, and the C ABI's b3_verify_multiple_locate state rules underneath.
// Signatures are synthesised with the library's input helpers (pk = [sk]G1, sig = [sk]H(msg)).  Needs an sm_100 device;
// exit code 0 = all checks passed.
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
    const int n = 6;
    std::vector<std::string> msgs;
    std::vector<AggregateSignature> sigs(n);
    std::vector<AggregatePublicKey> apks(n);
    for (int j = 0; j < n; j++) {
        Keypair k1 = keypair(3000 + 13 * j), k2 = keypair(5000 + 29 * j);
        msgs.push_back("per set " + std::to_string(j));
        Signature s1 = sign(k1, msgs[j]), s2 = sign(k2, msgs[j]);
        sigs[j] = AggregateSignature::aggregate({&s1, &s2});
        apks[j] = AggregatePublicKey::into_aggregate({k1.pk, k2.pk}).value;
    }
    auto sets_of = [&](const std::vector<AggregateSignature>& sg, const std::vector<std::string>& ms) {
        std::vector<AggregateSignature::Set> v;
        for (int j = 0; j < n; j++) v.push_back({&sg[j], &apks[j], bytes(ms[j]), ms[j].size()});
        return v;
    };
    {   // every set valid: all true, one 8-byte draw per set
        CountingRng rng(1);
        auto sets = sets_of(sigs, msgs);
        std::vector<bool> v = AggregateSignature::verify_multiple_aggregate_signatures_per_set(rng, sets.begin(), sets.end());
        CHECK(v == std::vector<bool>(n, true));
        CHECK(rng.consumed == n * 8);
    }
    {   // a tampered message (set 1) and another set's signature (set 4): exactly those two are false
        CountingRng rng(2);
        std::vector<std::string> tampered = msgs;
        tampered[1][0] ^= 1;
        std::vector<AggregateSignature> swapped = sigs;
        swapped[4] = sigs[5];
        auto sets = sets_of(swapped, tampered);
        std::vector<bool> v = AggregateSignature::verify_multiple_aggregate_signatures_per_set(rng, sets.begin(), sets.end());
        std::vector<bool> want(n, true);
        want[1] = want[4] = false;
        CHECK(v == want);
        CHECK(rng.consumed == n * 8);
        // the batch entry agrees, and the C ABI's locate after it returns the same verdicts again
        CountingRng rng2(2);
        CHECK(!AggregateSignature::verify_multiple_aggregate_signatures(rng2, sets.begin(), sets.end()));
        int32_t valid[n];
        size_t n_bad = 0;
        CHECK(b3_verify_multiple_locate(detail::ctx(), n, valid, &n_bad) == B3_OK && n_bad == 2);
        for (int j = 0; j < n; j++) CHECK((valid[j] != 0) == want[j]);
        CHECK(b3_verify_multiple_locate(detail::ctx(), n - 1, valid, &n_bad) == B3_ERR_ARG);            // wrong n
        CHECK(std::string(b3_last_error(detail::ctx())).find("locate") != std::string::npos);
    }
    {   // after any other call on the context, locate is refused
        (void)keypair(7);                                                      // b3_g1_mul_gen
        int32_t valid[n];
        CHECK(b3_verify_multiple_locate(detail::ctx(), n, valid, nullptr) == B3_ERR_ARG);
    }
    {   // empty batch: no verdicts, nothing drawn
        CountingRng rng(4);
        std::vector<AggregateSignature::Set> none;
        CHECK(AggregateSignature::verify_multiple_aggregate_signatures_per_set(rng, none.begin(), none.end()).empty());
        CHECK(rng.consumed == 0);
    }
    if (failures) std::printf("%d check(s) FAILED\n", failures);
    else std::printf("all checks passed\n");
    return failures ? 1 : 0;
}
