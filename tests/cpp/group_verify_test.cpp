// tests/cpp/group_verify_test.cpp — the C++ host layer's grouped call (include/lhb200.hpp:
// bls::verify_signature_set_groups): one verdict per group of SignatureSets, each equal to verify_signature_sets on that
// group alone.  Vectors as host_mirror_test.cpp (pk48 | msg32 | sig96 records, at least 12).
// Exit codes: 0 all good, 2 no usable GPU (the library has no CPU fallback), 1 a check failed.
#include <cstdio>
#include <vector>
#include "lhb200.hpp"

using namespace lhb200;

#define CHECK(c)                                                         \
    do {                                                                 \
        if (!(c)) { std::fprintf(stderr, "CHECK FAILED %s:%d: %s\n", __FILE__, __LINE__, #c); return 1; } \
    } while (0)

int main(int argc, char** argv) {
    if (lhb200_init(0) != LHB200_OK) {
        std::fprintf(stderr, "no device: %s\n", lhb200_last_error());
        return 2;
    }
    if (argc < 2) return 1;
    std::FILE* f = std::fopen(argv[1], "rb");
    if (!f) return 1;
    std::vector<bls::PublicKey> pks;
    std::vector<bls::Signature> sigs;
    std::vector<Hash256> msgs;
    uint8_t rec[176];
    while (std::fread(rec, 1, sizeof rec, f) == sizeof rec) {
        pks.push_back(bls::PublicKey::deserialize(rec, 48));
        Hash256 m;
        std::memcpy(m.data(), rec + 48, 32);
        msgs.push_back(m);
        sigs.push_back(bls::Signature::deserialize(rec + 80, 96));
    }
    std::fclose(f);
    CHECK(pks.size() >= 12);
    auto set = [&](size_t i) { return bls::SignatureSet::single_pubkey(sigs[i], pks[i], msgs[i]); };
    bls::SignatureSet tampered = set(3);
    tampered.message[0] ^= 1;
    bls::SignatureSet swapped = set(9);
    swapped.signature = &sigs[10];
    const bls::Signature empty = bls::Signature::empty();
    bls::SignatureSet empty_sig = set(11);
    empty_sig.signature = &empty;
    const std::vector<std::vector<bls::SignatureSet>> groups = {
        {set(0)}, {set(1), set(2)}, {}, {tampered}, {set(4), set(5), set(6), set(7), set(8)}, {set(2), swapped}, {empty_sig},
    };
    const std::vector<bool> got = bls::verify_signature_set_groups(groups);
    const std::vector<bool> want = {true, true, false, false, true, false, false};
    CHECK(got == want);
    for (size_t g = 0; g < groups.size(); g++)   // each verdict is the single-verdict call on that group alone
        CHECK(got[g] == bls::verify_signature_sets(groups[g].begin(), groups[g].end()));
    CHECK(bls::verify_signature_set_groups({}).empty());
    std::vector<std::vector<bls::SignatureSet>> per_set;
    for (size_t i = 0; i < pks.size(); i++) per_set.push_back({set(i)});
    const std::vector<bool> all = bls::verify_signature_set_groups(per_set);
    CHECK(all.size() == pks.size());
    for (bool v : all) CHECK(v);
    std::printf("OK %zu groups\n", groups.size() + per_set.size());
    return 0;
}
