// lhb200.hpp — header-only C++ host layer above the C ABI (include/lhb200.h), mirroring the reference's Rust
// surface for the two hot paths so that C++ callers (and the parity tests) read like Lighthouse code:
//
//   lhb200::bls::{PublicKey, Signature, AggregateSignature, SignatureSet, verify_signature_sets}
//        <-> crypto/bls/src/{generic_public_key.rs:46-102, generic_signature.rs:49-150,
//            generic_aggregate_signature.rs:60-235, generic_signature_set.rs:61-121, impls/blst.rs:37-119}
//   lhb200::tree_hash::{merkle_root, mix_in_length, hash32_concat, BeaconStateDeneb::update_tree_hash_cache}
//        <-> tree_hash crate call sites (crypto/bls/src/macros.rs:24), consensus/types/src/beacon_state.rs:2031-2038
//   lhb200::merkle_proof::{MerkleTree, verify_merkle_proof}
//        <-> consensus/merkle_proof/src/lib.rs:68-99,290-324,357-389
//
// (The reference is Rust; there is no Rust toolchain in the build image, so the compiled host layer is C++.  The
//  Rust shim is shown in INTEGRATION.md.)  Errors: decode failures throw lhb200::Error (bls::Error in the
//  reference); verify* return bool and fail closed on any library status.
#pragma once
#include <array>
#include <cstdint>
#include <cstring>
#include <stdexcept>
#include <string>
#include <vector>
#include "lhb200.h"

namespace lhb200 {

struct Error : std::runtime_error {
    int32_t code;
    Error(int32_t c, const std::string& what) : std::runtime_error(what + ": " + lhb200_last_error()), code(c) {}
};
inline void check(int32_t rc, const char* where) {
    if (rc != LHB200_OK) throw Error(rc, where);
}
inline void init(int device = 0) { check(lhb200_init(device), "lhb200_init"); }

using Hash256 = std::array<uint8_t, 32>;

namespace bls {

constexpr size_t PUBLIC_KEY_BYTES_LEN = 48, PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN = 96, SIGNATURE_BYTES_LEN = 96;

/// GenericPublicKey: validated at deserialize (subgroup, not infinity — generic_public_key.rs:86-94, blst.rs:130-140).
class PublicKey {
  public:
    static PublicKey deserialize(const uint8_t* bytes, size_t len) {
        if (len != PUBLIC_KEY_BYTES_LEN) throw Error(LHB200_EINVAL, "InvalidByteLength");
        PublicKey pk;
        uint8_t st = 0;
        check(lhb200_g1_decompress_validate(bytes, 1, pk.uncompressed_.data(), &st), "lhb200_g1_decompress_validate");
        if (st == 1) throw Error(LHB200_EDECODE, "InvalidInfinityPublicKey");
        if (st != 0) throw Error(LHB200_EDECODE, "BlstError(key_validate)");
        std::memcpy(pk.compressed_.data(), bytes, 48);
        return pk;
    }
    /// TPublicKey::deserialize_uncompressed (blst.rs:142-150; generic_public_key.rs:96-102): curve check, no subgroup
    /// check, infinity rejected like deserialize.
    static PublicKey deserialize_uncompressed(const uint8_t* bytes, size_t len) {
        if (len != PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN) throw Error(LHB200_EINVAL, "InvalidByteLength");
        PublicKey pk;
        uint8_t st = 0;
        check(lhb200_g1_deserialize_uncompressed(bytes, 1, pk.compressed_.data(), &st), "lhb200_g1_deserialize_uncompressed");
        if (st == 1) throw Error(LHB200_EDECODE, "InvalidInfinityPublicKey");
        if (st != 0) throw Error(LHB200_EDECODE, "BlstError(bad G1 encoding)");
        std::memcpy(pk.uncompressed_.data(), bytes, 96);
        return pk;
    }
    const std::array<uint8_t, 48>& serialize() const { return compressed_; }
    const std::array<uint8_t, 96>& serialize_uncompressed() const { return uncompressed_; }
    bool operator==(const PublicKey& o) const { return compressed_ == o.compressed_; }

  private:
    friend class AggregatePublicKey;
    std::array<uint8_t, 48> compressed_{};
    std::array<uint8_t, 96> uncompressed_{};
};

/// GenericAggregatePublicKey::aggregate (generic_aggregate_public_key.rs:9-15, blst.rs:178-184): the sum of validated
/// keys; an empty list is an error, an infinite sum is reported like the reference's `InvalidInfinityPublicKey`.
class AggregatePublicKey {
  public:
    static AggregatePublicKey aggregate(const std::vector<const PublicKey*>& pks) {
        if (pks.empty()) throw Error(LHB200_EINVAL, "EmptyAggregate");
        std::vector<uint8_t> flat;
        for (const PublicKey* pk : pks) flat.insert(flat.end(), pk->uncompressed_.begin(), pk->uncompressed_.end());
        AggregatePublicKey a;
        check(lhb200_g1_aggregate(flat.data(), static_cast<uint32_t>(pks.size()), a.pk_.compressed_.data(),
                                  a.pk_.uncompressed_.data()), "lhb200_g1_aggregate");
        if (a.pk_.compressed_[0] & 0x40) throw Error(LHB200_EDECODE, "InvalidInfinityPublicKey");
        return a;
    }
    const PublicKey& to_public_key() const { return pk_; }

  private:
    PublicKey pk_;
};

/// GenericSignature / GenericAggregateSignature: canonical bytes; all-zero = the "empty" signature (point None).
class Signature {
  public:
    static Signature empty() { return Signature(); }
    static Signature infinity() {
        Signature s;
        s.bytes_[0] = 0xc0;
        return s;
    }
    static Signature deserialize(const uint8_t* bytes, size_t len) {
        if (len != SIGNATURE_BYTES_LEN) throw Error(LHB200_EINVAL, "InvalidByteLength");
        Signature s;
        std::memcpy(s.bytes_.data(), bytes, 96);
        if (s.is_empty()) return s;
        uint8_t xy[192], st = 0;
        check(lhb200_g2_decompress(bytes, 1, xy, &st), "lhb200_g2_decompress");
        if (st == 2) throw Error(LHB200_EDECODE, "BlstError(bad G2 encoding)");
        return s;
    }
    const std::array<uint8_t, 96>& serialize() const { return bytes_; }
    bool is_empty() const {
        for (uint8_t b : bytes_)
            if (b) return false;
        return true;
    }
    bool is_infinity() const {
        if (bytes_[0] != 0xc0) return false;
        for (size_t i = 1; i < 96; i++)
            if (bytes_[i]) return false;
        return true;
    }

  private:
    std::array<uint8_t, 96> bytes_{};
};
struct SignatureSet;
/// GenericAggregateSignature (generic_aggregate_signature.rs:60-235): a Signature that can absorb others.
/// add_assign / add_assign_aggregate are point additions on the device (blst.rs:230-237); the infinity encoding is the
/// identity and the "empty" (all-zero) aggregate takes the value of the first signature added (:111-124).
class AggregateSignature : public Signature {
  public:
    AggregateSignature() : Signature(Signature::infinity()) {}
    explicit AggregateSignature(const Signature& s) : Signature(s) {}
    static AggregateSignature deserialize(const uint8_t* bytes, size_t len) {
        return AggregateSignature(Signature::deserialize(bytes, len));
    }
    void add_assign(const Signature& other) {
        if (other.is_empty()) return;
        if (is_empty()) { static_cast<Signature&>(*this) = other; return; }
        uint8_t two[192], out[96];
        std::memcpy(two, serialize().data(), 96);
        std::memcpy(two + 96, other.serialize().data(), 96);
        check(lhb200_g2_aggregate(two, 2, out), "lhb200_g2_aggregate");
        static_cast<Signature&>(*this) = Signature::deserialize(out, 96);
    }
    void add_assign_aggregate(const AggregateSignature& other) { add_assign(other); }
    /// AggregateSignature::aggregate of many signatures in ONE device call
    static AggregateSignature aggregate(const std::vector<const Signature*>& sigs) {
        std::vector<uint8_t> flat;
        for (const Signature* s : sigs)
            if (!s->is_empty()) flat.insert(flat.end(), s->serialize().begin(), s->serialize().end());
        uint8_t out[96];
        check(lhb200_g2_aggregate(flat.empty() ? nullptr : flat.data(), static_cast<uint32_t>(flat.size() / 96), out),
              "lhb200_g2_aggregate");
        return AggregateSignature(Signature::deserialize(out, 96));
    }
    /// aggregate_verify (generic_aggregate_signature.rs:212-235, blst.rs:263-273): distinct messages, one key each
    bool aggregate_verify(const std::vector<Hash256>& msgs, const std::vector<const PublicKey*>& pks) const {
        if (msgs.empty() || msgs.size() != pks.size() || is_empty()) return false;
        std::vector<uint8_t> m, k;
        for (const Hash256& h : msgs) m.insert(m.end(), h.begin(), h.end());
        for (const PublicKey* pk : pks) k.insert(k.end(), pk->serialize_uncompressed().begin(), pk->serialize_uncompressed().end());
        uint8_t ok = 0;
        const int32_t rc = lhb200_aggregate_verify(serialize().data(), m.data(), k.data(), static_cast<uint32_t>(msgs.size()), &ok);
        return rc == LHB200_OK && ok == 1;
    }
};

/// GenericSignatureSet {signature, signing_keys, message} — borrows, like the Cow<'a, ..> fields of the reference.
struct SignatureSet {
    const Signature* signature;   // a Signature or an AggregateSignature (GenericSignatureSet holds the aggregate form)
    std::vector<const PublicKey*> signing_keys;
    Hash256 message;
    static SignatureSet single_pubkey(const Signature& s, const PublicKey& pk, const Hash256& m) {
        return SignatureSet{&s, {&pk}, m};
    }
    static SignatureSet multiple_pubkeys(const Signature& s, std::vector<const PublicKey*> pks, const Hash256& m) {
        return SignatureSet{&s, std::move(pks), m};
    }
    bool verify() const;
};

/// bls::verify_signature_sets (impls/blst.rs:37-119): flatten to SoA, one C-ABI call, fail closed.
template <class It>
inline bool verify_signature_sets(It begin, It end) {
    std::vector<uint8_t> sigs, msgs, pks;
    std::vector<uint32_t> offs{0};
    for (It it = begin; it != end; ++it) {
        const SignatureSet& set = *it;
        sigs.insert(sigs.end(), set.signature->serialize().begin(), set.signature->serialize().end());
        msgs.insert(msgs.end(), set.message.begin(), set.message.end());
        for (const PublicKey* pk : set.signing_keys)
            pks.insert(pks.end(), pk->serialize_uncompressed().begin(), pk->serialize_uncompressed().end());
        offs.push_back(static_cast<uint32_t>(pks.size() / 96));
    }
    const uint32_t n = static_cast<uint32_t>(offs.size() - 1);
    if (n == 0) return false;  // blst.rs:42-44
    uint8_t ok = 0;
    const int32_t rc = lhb200_verify_signature_sets(sigs.data(), msgs.data(), pks.empty() ? nullptr : pks.data(),
                                                    offs.data(), nullptr, n, &ok, nullptr);
    return rc == LHB200_OK && ok == 1;
}
inline bool SignatureSet::verify() const { return verify_signature_sets(this, this + 1); }

/// Many independent verify_signature_sets calls in one device pass (lhb200_verify_signature_set_groups):
/// result[g] == verify_signature_sets(groups[g]); an empty group is false.  Fails closed per group: any library error
/// makes every element false.
inline std::vector<bool> verify_signature_set_groups(const std::vector<std::vector<SignatureSet>>& groups) {
    std::vector<uint8_t> sigs, msgs, pks;
    std::vector<uint32_t> offs{0}, goffs{0};
    for (const std::vector<SignatureSet>& group : groups) {
        for (const SignatureSet& set : group) {
            sigs.insert(sigs.end(), set.signature->serialize().begin(), set.signature->serialize().end());
            msgs.insert(msgs.end(), set.message.begin(), set.message.end());
            for (const PublicKey* pk : set.signing_keys)
                pks.insert(pks.end(), pk->serialize_uncompressed().begin(), pk->serialize_uncompressed().end());
            offs.push_back(static_cast<uint32_t>(pks.size() / 96));
        }
        goffs.push_back(static_cast<uint32_t>(offs.size() - 1));
    }
    const uint32_t n_groups = static_cast<uint32_t>(groups.size());
    std::vector<uint8_t> ok(n_groups, 0);
    const int32_t rc = lhb200_verify_signature_set_groups(sigs.data(), msgs.data(), pks.empty() ? nullptr : pks.data(),
                                                          offs.data(), nullptr, static_cast<uint32_t>(offs.size() - 1),
                                                          goffs.data(), n_groups, ok.data(), nullptr);
    std::vector<bool> out(n_groups, false);
    if (rc == LHB200_OK)
        for (uint32_t g = 0; g < n_groups; g++) out[g] = ok[g] == 1;
    return out;
}

/// fast_aggregate_verify / eth_fast_aggregate_verify (generic_aggregate_signature.rs:187-210)
inline bool fast_aggregate_verify(const Signature& sig, const Hash256& msg, const std::vector<const PublicKey*>& pks) {
    if (pks.empty()) return false;
    return SignatureSet::multiple_pubkeys(sig, pks, msg).verify();
}
inline bool eth_fast_aggregate_verify(const Signature& sig, const Hash256& msg, const std::vector<const PublicKey*>& pks) {
    if (pks.empty() && sig.is_infinity()) return true;
    return fast_aggregate_verify(sig, msg, pks);
}

/// ParallelSignatureSets (state_processing/src/per_block_processing/block_signature_verifier.rs:84-96,392-418):
/// accumulate the sets of 1..N blocks, verify them with one batch call.
class ParallelSignatureSets {
  public:
    void push(SignatureSet set) { sets_.push_back(std::move(set)); }
    size_t size() const { return sets_.size(); }
    bool verify() const { return verify_signature_sets(sets_.begin(), sets_.end()); }

  private:
    std::vector<SignatureSet> sets_;
};

}  // namespace bls

namespace tree_hash {

constexpr size_t BYTES_PER_CHUNK = 32;

inline Hash256 hash32_concat(const Hash256& a, const Hash256& b) {
    uint8_t in[64];
    std::memcpy(in, a.data(), 32);
    std::memcpy(in + 32, b.data(), 32);
    Hash256 out;
    check(lhb200_hash_pairs(in, out.data(), 1), "lhb200_hash_pairs");
    return out;
}
/// tree_hash::merkle_root(bytes, minimum_leaf_count)
inline Hash256 merkle_root(const uint8_t* bytes, size_t len, size_t minimum_leaf_count = 0) {
    const size_t n = len ? (len + 31) / 32 : 1;
    std::vector<uint8_t> padded(n * 32, 0);
    std::memcpy(padded.data(), bytes, len);
    size_t leaves = n > minimum_leaf_count ? n : minimum_leaf_count;
    uint32_t depth = 0;
    while ((size_t(1) << depth) < leaves) depth++;
    Hash256 out;
    check(lhb200_merkleize(padded.data(), n, depth, out.data()), "lhb200_merkleize");
    return out;
}
inline Hash256 mix_in_length(const Hash256& root, uint64_t length) {
    Hash256 out;
    check(lhb200_mix_in_length(root.data(), length, out.data()), "lhb200_mix_in_length");
    return out;
}
/// BeaconState::update_tree_hash_cache for BeaconStateDeneb SSZ bytes (cold).
inline Hash256 beacon_state_root_deneb(const uint8_t* ssz, size_t len) {
    Hash256 out;
    check(lhb200_beacon_state_root_deneb(ssz, len, out.data(), nullptr), "lhb200_beacon_state_root_deneb");
    return out;
}

/// the same for any post-Altair fork id (LHB200_FORK_ALTAIR .. LHB200_FORK_ELECTRA; beacon_state.rs:224-571)
inline Hash256 beacon_state_root(const uint8_t* ssz, size_t len, int32_t fork) {
    Hash256 out;
    check(lhb200_beacon_state_root(ssz, len, fork, out.data(), nullptr), "lhb200_beacon_state_root");
    return out;
}

/// BeaconBlock::canonical_root (beacon_block.rs:158-160) for BeaconBlockDeneb SSZ bytes.
inline Hash256 beacon_block_root_deneb(const uint8_t* ssz, size_t len, Hash256* body_root = nullptr) {
    Hash256 out;
    check(lhb200_beacon_block_root_deneb(ssz, len, out.data(), body_root ? body_root->data() : nullptr),
          "lhb200_beacon_block_root_deneb");
    return out;
}

/// canonical_root of one BeaconBlock / BlindedBeaconBlock of any fork from Altair to Deneb (beacon_block.rs:41-90)
inline Hash256 beacon_block_root(const uint8_t* ssz, size_t len, int32_t fork, bool blinded = false, Hash256* body_root = nullptr) {
    Hash256 out;
    const uint64_t offs[2] = {0, len};
    check(lhb200_beacon_block_roots(ssz, offs, 1, fork, blinded ? 1 : 0, out.data(), body_root ? body_root->data() : nullptr),
          "lhb200_beacon_block_roots");
    return out;
}

}  // namespace tree_hash

namespace swap_or_not_shuffle {
/// shuffle_list(input, rounds, seed, forwards) -> Option<Vec<usize>> (shuffle_list.rs:79): empty vector = None.
inline std::vector<uint64_t> shuffle_list(const std::vector<uint64_t>& input, uint8_t rounds, const Hash256& seed,
                                          bool forwards) {
    std::vector<uint64_t> out(input.size());
    const int32_t rc = lhb200_shuffle_list(input.data(), input.size(), rounds, seed.data(), forwards ? 1 : 0, out.data());
    if (rc == LHB200_EINVAL) return {};
    check(rc, "lhb200_shuffle_list");
    return out;
}
}  // namespace swap_or_not_shuffle

namespace merkle_proof {

/// MerkleTree::create(leaves, depth) — right-sparse fixed-depth tree.
class MerkleTree {
  public:
    MerkleTree(std::vector<Hash256> leaves, uint32_t depth) : leaves_(std::move(leaves)), depth_(depth) {
        if (depth > 32 || leaves_.size() > (uint64_t(1) << depth)) throw Error(LHB200_EINVAL, "MerkleTreeError::DepthTooSmall");
    }
    static MerkleTree create(std::vector<Hash256> leaves, uint32_t depth) { return MerkleTree(std::move(leaves), depth); }
    Hash256 hash() const { return proof(0).first; }
    /// generate_proof(index, depth) -> (leaf, bottom-up branch)
    std::pair<Hash256, std::vector<Hash256>> generate_proof(uint64_t index) const {
        auto pr = proof(index);
        Hash256 leaf{};
        if (index < leaves_.size()) leaf = leaves_[index];
        return {leaf, pr.second};
    }

  private:
    std::pair<Hash256, std::vector<Hash256>> proof(uint64_t index) const {
        Hash256 root;
        std::vector<Hash256> branch(depth_);
        check(lhb200_merkle_tree_proof(leaves_.empty() ? nullptr : leaves_[0].data(), leaves_.size(), depth_, index,
                                       root.data(), depth_ ? branch[0].data() : nullptr),
              "lhb200_merkle_tree_proof");
        return {root, branch};
    }
    std::vector<Hash256> leaves_;
    uint32_t depth_;
};
inline bool verify_merkle_proof(const Hash256& leaf, const std::vector<Hash256>& branch, uint32_t depth, uint64_t index,
                                const Hash256& root) {
    if (branch.size() != depth) return false;  // lib.rs:364
    uint8_t ok = 0;
    const int32_t rc = lhb200_verify_merkle_proofs(leaf.data(), depth ? branch[0].data() : leaf.data(), depth, &index,
                                                   root.data(), 1, &ok);
    return rc == LHB200_OK && ok == 1;
}

}  // namespace merkle_proof
}  // namespace lhb200
