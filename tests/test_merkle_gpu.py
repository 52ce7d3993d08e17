"""GPU parity tests for the tree-hash path: CUDA library (through the C ABI) vs the CPU oracle and the
reference's golden vectors.  Bit-exact (32-byte digests)."""
import hashlib
import struct

import numpy as np
import pytest

from tests import oracle_lib as O

pytestmark = pytest.mark.gpu


def rb(rng, n):
    return rng.integers(0, 256, n, dtype=np.uint8).tobytes()


def test_zero_hashes(gpu):
    from lighthouse_b200 import tree_hash as T
    for d in range(0, 65):
        assert T.zero_hash(d) == O.zero_hash(d)


@pytest.mark.parametrize("n", [1, 2, 31, 256, 257, 10_000])
def test_hash_pairs(gpu, n):
    from lighthouse_b200 import tree_hash as T
    d = rb(np.random.default_rng(n), 64 * n)
    got = T.hash_pairs(d)
    assert got == O.hash_pairs(d)
    assert got[:32] == hashlib.sha256(d[:64]).digest()


@pytest.mark.parametrize("n,depth", [(0, 0), (0, 7), (1, 0), (1, 1), (1, 40), (2, 1), (3, 2), (5, 3), (7, 30), (8, 3),
                                     (9, 4), (9, 40), (16, 4), (17, 5), (255, 8), (256, 8), (257, 9), (2047, 11),
                                     (2048, 11), (2049, 12), (2049, 40), (4097, 13), (100_003, 17), (100_003, 38),
                                     (1 << 16, 16), (300_000, 35)])
def test_merkleize_vs_oracle(gpu, n, depth):
    from lighthouse_b200 import tree_hash as T
    c = rb(np.random.default_rng(n * 977 + depth), 32 * n)
    assert T.merkleize_chunks(c, depth) == O.merkleize(c, depth)


def test_merkle_root_and_mix_in_length(gpu):
    from lighthouse_b200 import tree_hash as T
    rng = np.random.default_rng(5)
    pk, sig = rb(rng, 48), rb(rng, 96)
    assert T.merkle_root(pk, 0) == O.merkleize_bytes(pk, 1)       # 48-byte blob (bls/src/macros.rs:18-25)
    assert T.merkle_root(sig, 0) == O.merkleize_bytes(sig, 2)     # 96-byte blob: 3 chunks padded to 4
    r = rb(rng, 32)
    for ln in (0, 1, 500_000, (1 << 40) - 1):
        assert T.mix_in_length(r, ln) == hashlib.sha256(r + struct.pack("<Q", ln) + b"\0" * 24).digest()


@pytest.mark.parametrize("net", ["sepolia", "gnosis", "mainnet"])
def test_genesis_validators_root_golden(gpu, net):
    """hash_tree_root(validators) of the reference's vendored genesis states == genesis_validators_root."""
    from lighthouse_b200 import tree_hash as T
    meta = O.golden_json("genesis_validators.json")[net]
    ssz = O.golden_validators(net)
    lo = meta.get("stored_from", 0)
    if lo:   # validators [lo, n) stored, with the root of the subtree over [0, lo)
        d = lo.bit_length() - 1
        node = T.hash_pairs(bytes.fromhex(meta["left_subtree_root"]) + T.merkleize_chunks(T.validator_roots(ssz), d))
        for lvl in range(d + 1, 40):
            node = T.hash_pairs(node + T.zero_hash(lvl))
        assert T.mix_in_length(node, meta["n_validators"]).hex() == meta["genesis_validators_root"]
        assert T.validators_root(ssz) == O.validators_root(ssz)
    else:
        assert T.validators_root(ssz).hex() == meta["genesis_validators_root"]
    assert T.validator_roots(ssz) == O.validator_roots(ssz)


@pytest.mark.parametrize("n", [0, 1, 255, 256, 257, 1000])
def test_validators_root_ragged(gpu, n):
    from lighthouse_b200 import tree_hash as T
    from lighthouse_b200.synthetic import validators_ssz
    ssz = validators_ssz(n, np.random.default_rng(n))
    assert T.validators_root(ssz) == O.validators_root(ssz)


def test_deposit_roots_golden(gpu):
    from lighthouse_b200 import tree_hash as T
    for d in O.golden_json("deposit_data.json"):
        pk = bytes.fromhex(d["pubkey"]); wc = bytes.fromhex(d["withdrawal_credentials"])
        amount = struct.pack("<Q", d["amount"]) + b"\0" * 24
        sig = bytes.fromhex(d["signature"])
        pk_root, sig_root = T.merkle_root(pk), T.merkle_root(sig)
        assert T.merkleize_chunks(pk_root + wc + amount, 2).hex() == d["deposit_message_root"]
        assert T.merkleize_chunks(pk_root + wc + amount + sig_root, 2).hex() == d["deposit_data_root"]


@pytest.mark.parametrize("nv,kw", [(0, dict(all_default=True)), (1, {}), (300, dict(n_hist_roots=5, n_votes=7,
                                                                                     n_summaries=3)),
                                   (5000, dict(all_default=True)), (16_384, {}), (70_001, dict(extra_data_len=32))])
def test_beacon_state_root_vs_oracle(gpu, nv, kw):
    from lighthouse_b200 import tree_hash as T
    from lighthouse_b200.synthetic import beacon_state_deneb_ssz
    ssz = beacon_state_deneb_ssz(nv, seed=nv + 1, **kw)
    want_root, want_fields = O.beacon_state_root_deneb(ssz)
    got_root, got_fields = T.beacon_state_root_deneb(ssz, want_field_roots=True)
    for i, (g, w) in enumerate(zip(got_fields, want_fields)):
        assert g == w, f"field {i} root differs"
    assert got_root == want_root


def test_beacon_state_full_size_resident(gpu):
    """BASELINE configs[1]: 500k-validator Deneb state; resident handle re-hashes to the same digest
    (idempotence) and matches the multi-threaded oracle."""
    from lighthouse_b200 import tree_hash as T
    from lighthouse_b200.synthetic import beacon_state_deneb_ssz
    ssz = beacon_state_deneb_ssz(500_000, seed=42)
    O.set_threads(O.hw_threads())
    want, _ = O.beacon_state_root_deneb(ssz)
    O.set_threads(1)
    st = T.ResidentState(ssz)
    r1 = st.root()
    r2 = st.root()
    units = st.hash_units
    st.release()
    assert r1 == r2 == want
    assert abs(units - 4_873_001) < 20_000, units  # SURVEY §8d algorithmic unit count (±small-field variation)


def test_malformed_state_rejected(gpu):
    from lighthouse_b200 import tree_hash as T, Lhb200Error
    from lighthouse_b200.synthetic import beacon_state_deneb_ssz
    ssz = bytearray(beacon_state_deneb_ssz(10, seed=1))
    ssz[524552:524556] = struct.pack("<I", 5)  # validators offset before the fixed part
    with pytest.raises(Lhb200Error):
        T.beacon_state_root_deneb(bytes(ssz))
    with pytest.raises(Lhb200Error):
        T.beacon_state_root_deneb(bytes(100))


def test_merkle_tree_create_and_proofs(gpu):
    """MerkleTree::create / generate_proof / verify_merkle_proof (merkle_proof/src/lib.rs tests :412-568)."""
    from lighthouse_b200.merkle_proof import MerkleTree, verify_merkle_proof, verify_merkle_proofs
    rng = np.random.default_rng(11)
    for depth, n in [(0, 1), (1, 1), (1, 2), (3, 5), (5, 32), (12, 6), (17, 100), (32, 9), (4, 0)]:
        leaves = [rb(rng, 32) for _ in range(n)]
        t = MerkleTree.create(leaves, depth)
        want_root = O.merkleize(b"".join(leaves), depth)
        assert t.hash() == want_root
        for idx in sorted({0, max(n - 1, 0), min(n, (1 << depth) - 1)}):
            leaf, br = t.generate_proof(idx, depth)
            wr, wb = O.merkle_tree_proof(leaves, depth, idx)
            assert br == wb and wr == want_root
            assert verify_merkle_proof(leaf, br, depth, idx, want_root)
            if depth:
                assert not verify_merkle_proof(leaf, br, depth, idx ^ 1, want_root) or br[0] == leaf
                bad = [bytes(32)] + br[1:]
                if bad != br:
                    assert not verify_merkle_proof(leaf, bad, depth, idx, want_root)
            assert not verify_merkle_proof(leaf, br[:-1], depth, idx, want_root) if depth else True
    # depth 0: verify_merkle_proof(leaf, [], 0, idx, root) <=> leaf == root   (lib.rs:562-568)
    x = rb(rng, 32)
    assert verify_merkle_proof(x, [], 0, 0, x) and not verify_merkle_proof(x, [], 0, 0, rb(rng, 32))
    # batch
    leaves = [rb(rng, 32) for _ in range(300)]
    t = MerkleTree.create(leaves, 10)
    root = t.hash()
    proofs = [t.generate_proof(i)[1] for i in range(0, 300, 37)]
    idxs = list(range(0, 300, 37))
    oks = verify_merkle_proofs([leaves[i] for i in idxs], proofs, 10, idxs, [root] * len(idxs))
    assert all(oks)
    oks = verify_merkle_proofs([leaves[i] for i in idxs], proofs, 10, [i + 1 for i in idxs], [root] * len(idxs))
    assert not any(oks)


@pytest.mark.parametrize("world", [2, 4, 8])
@pytest.mark.parametrize("nv", [70_001, 300])
def test_sharded_state_root_equals_full(gpu, world, nv):
    """SURVEY §8e: one state split into `world` leaf ranges (simulated in one process): per-rank subtree roots,
    one all-gather, combine -> the same 32-byte root as the single-GPU path and the oracle."""
    from lighthouse_b200 import tree_hash as T
    from lighthouse_b200.synthetic import beacon_state_deneb_ssz
    ssz = beacon_state_deneb_ssz(nv, seed=nv)
    want, _ = O.beacon_state_root_deneb(ssz)
    shards = [T.ShardedState(ssz, r, world) for r in range(world)]
    parts = [s.shard_roots() for s in shards]
    assert len({len(p) for p in parts}) == 1
    gathered = b"".join(parts)                      # what the all-gather delivers (rank-major)
    for s in shards:
        assert s.combine(gathered) == want
        s.release()


def test_resident_state_patch_matches_oracle(gpu):
    """SURVEY §8f-3 (warm path): mutate a staged state in place — validator records, balances, participation,
    randao mix, slot, latest_block_header, a checkpoint — and re-hash; must equal the oracle on the mutated SSZ."""
    from lighthouse_b200 import tree_hash as T, Lhb200Error
    from lighthouse_b200.synthetic import beacon_state_deneb_ssz
    rng = np.random.default_rng(8)
    ssz = bytearray(beacon_state_deneb_ssz(20_000, seed=77))
    st = T.ResidentState(bytes(ssz))
    assert st.root() == O.beacon_state_root_deneb(bytes(ssz))[0]
    o_val, o_bal = struct.unpack_from("<II", ssz, 524552)
    o_pp, o_cp = struct.unpack_from("<II", ssz, 2687248)
    edits = []
    for vi in (0, 123, 19_999):                                   # effective_balance + exit_epoch of 3 validators
        edits.append((o_val + 121 * vi + 80, struct.pack("<Q", 31_000_000_000 + vi)))
        edits.append((o_val + 121 * vi + 105, struct.pack("<Q", 4242 + vi)))
    edits.append((o_bal + 8 * 777, struct.pack("<Q", 123456789)))                       # one balance
    edits.append((o_bal + 8 * 1000, rb(rng, 8 * 64)))                                   # 64 consecutive balances
    edits.append((o_pp + 5000, bytes([7] * 100)))                                       # participation flags
    edits.append((524560 + 32 * 4097, rb(rng, 32)))                                     # one randao mix
    edits.append((40, struct.pack("<Q", 9_999_999)))                                    # slot
    edits.append((64, rb(rng, 112)))                                                    # latest_block_header
    edits.append((2687297, rb(rng, 40)))                                                # current_justified_checkpoint
    edits.append((2687256, bytes([0x05])))                                              # justification_bits
    for off, data in edits:
        ssz[off:off + len(data)] = data
        st.patch(off, data)
    want, want_fields = O.beacon_state_root_deneb(bytes(ssz))
    got, got_fields = st.root(want_field_roots=True)
    for i, (g, w) in enumerate(zip(got_fields, want_fields)):
        assert g == w, f"field {i}"
    assert got == want
    with pytest.raises(Lhb200Error):
        st.patch(524552, b"\\0\\0\\0\\0")                                                  # offset table: refused
    st.release()


@pytest.mark.parametrize("n_validators", [20_000, 300_001])
def test_incremental_state_root_matches_oracle(gpu, n_validators):
    """Warm path with resident level arrays (lhb200_state_enable_incremental): several rounds of slot-like mutations —
    scattered validator records, balances, participation flags, inactivity scores, one randao mix, block/state roots,
    slashings, small fixed fields — each followed by a root that re-hashes only dirty paths; every root and every field
    root must equal the oracle on the mutated SSZ.  A patch to a list without a resident tree (historical_roots)
    falls back to a cold root; the following round is warm again."""
    from lighthouse_b200 import tree_hash as T
    from lighthouse_b200.synthetic import beacon_state_deneb_ssz
    rng = np.random.default_rng(n_validators)
    ssz = bytearray(beacon_state_deneb_ssz(n_validators, seed=5))
    st = T.ResidentState(bytes(ssz))
    cold_units = st.hash_units
    st.enable_incremental()
    assert st.root() == O.beacon_state_root_deneb(bytes(ssz))[0]
    assert st.last_root_hashes == cold_units                        # first root after enabling is cold
    o_hist = struct.unpack_from("<I", ssz, 524464)[0]
    o_val, o_bal = struct.unpack_from("<II", ssz, 524552)
    o_pp, o_cp = struct.unpack_from("<II", ssz, 2687248)
    o_inact = struct.unpack_from("<I", ssz, 2687377)[0]

    pending = []

    def apply(off, data):
        ssz[off:off + len(data)] = data
        if rnd % 2:
            pending.append((off, data))          # odd rounds: one lhb200_state_patch_batch call for the whole slot
        else:
            st.patch(off, data)

    for rnd in range(4):
        for vi in rng.choice(n_validators, size=300, replace=False):          # effective balances / exit epochs
            apply(o_val + 121 * int(vi) + 80, struct.pack("<Q", int(rng.integers(1, 1 << 40))))
            if vi % 3 == 0:
                apply(o_val + 121 * int(vi) + 105, struct.pack("<Q", int(rng.integers(1, 1 << 30))))
        apply(o_val + 121 * (n_validators - 1) + 88, bytes([1]))              # slashed flag of the last validator
        for bi in rng.choice(n_validators, size=500, replace=False):
            apply(o_bal + 8 * int(bi), struct.pack("<Q", int(rng.integers(1, 1 << 45))))
        apply(o_cp + int(rng.integers(0, n_validators - 2000)), rb(rng, 2000))  # a committee's participation flags
        apply(o_pp + n_validators - 1, bytes([3]))                            # last (partial) chunk of a packed list
        apply(o_inact + 8 * int(rng.integers(0, n_validators)), struct.pack("<Q", rnd + 1))
        apply(524560 + 32 * int(rng.integers(0, 65536)), rb(rng, 32))         # randao mix
        apply(176 + 32 * int(rng.integers(0, 8192)), rb(rng, 32))             # block_roots[i]
        apply(262320 + 32 * int(rng.integers(0, 8192)), rb(rng, 32))          # state_roots[i]
        apply(2621712 + 8 * int(rng.integers(0, 8192)), struct.pack("<Q", int(rng.integers(1, 1 << 40))))  # slashings
        apply(40, struct.pack("<Q", 1000 + rnd))                              # slot
        apply(64, rb(rng, 112))                                               # latest_block_header
        if rnd == 2:
            apply(o_hist + 32, rb(rng, 32))                                   # historical_roots: no resident tree
        if pending:                                                           # later edits of the same bytes win:
            last = {}                                                         # keep the batch non-overlapping
            for off, data in pending:
                last[(off, len(data))] = data
            st.patch_batch([(o, d) for (o, _), d in last.items()])
            pending.clear()
        want, want_fields = O.beacon_state_root_deneb(bytes(ssz))
        got, got_fields = st.root(want_field_roots=True)
        for i, (g, w) in enumerate(zip(got_fields, want_fields)):
            assert g == w, f"round {rnd} field {i}"
        assert got == want
        if rnd == 2:
            assert st.last_root_hashes == cold_units                          # fell back to a cold root
        else:
            assert st.last_root_hashes < cold_units // 20                     # warm: dirty paths + tail only
    assert st.root() == O.beacon_state_root_deneb(bytes(ssz))[0]              # nothing dirty: tail only, same root
    st.release()


def test_merkle_hasher_attestation_key(gpu):
    """AttestationKey::tree_hash_root (naive_aggregation_pool.rs:44-58): MerkleHasher::with_leaves(2), write the data
    root, write the committee index -> H(data_root || le64(index) zero-padded)."""
    from lighthouse_b200 import tree_hash as T
    data_root = hashlib.sha256(b"attestation data").digest()
    got = T.MerkleHasher.with_leaves(2).write(data_root).write((37).to_bytes(8, "little")).finish()
    assert got == hashlib.sha256(data_root + (37).to_bytes(8, "little") + bytes(24)).digest()
    h = T.MerkleHasher.with_leaves(4).write(data_root)
    assert h.finish() == O.merkleize(data_root, 2)                      # right-sparse: zero-hash padding
    with pytest.raises(ValueError):
        T.MerkleHasher.with_leaves(1).write(data_root).write(b"\x01")


def test_signing_root_and_domain_helpers(gpu):
    """signing_root / compute_domain (signing_data.rs:27-35, chain_spec.rs:548-566) against hashlib and the
    synthetic generator's own CPU restatement."""
    from lighthouse_b200 import tree_hash as T
    from lighthouse_b200.synthetic import attester_domain, MAINNET_GVR
    dom = T.compute_domain(1, bytes.fromhex("04000000"), MAINNET_GVR)
    assert dom == attester_domain()
    roots = b"".join(hashlib.sha256(bytes([i])).digest() for i in range(50))
    got = T.signing_roots(roots, dom)
    for i in range(50):
        assert got[32 * i:32 * i + 32] == hashlib.sha256(roots[32 * i:32 * i + 32] + dom).digest()
    leaves = [hashlib.sha256(bytes([i])).digest() for i in range(5)]
    assert T.container_root(leaves) == O.merkleize(b"".join(leaves), 3)


@pytest.mark.parametrize("fork", ["altair", "bellatrix", "capella", "deneb", "electra"])
@pytest.mark.parametrize("nv,kw", [(0, {"all_default": True}), (37, {}), (1500, {"n_hist_roots": 3, "n_votes": 5, "n_summaries": 2})])
def test_beacon_state_root_every_post_altair_fork(gpu, fork, nv, kw):
    """BeaconState superstruct variants (consensus/types/src/beacon_state.rs:224-571) through the fork-parametrised
    describer: root and every field root against the GENERIC from-spec merkleization of tests/ssz_spec.py over the
    decoded value (type descriptors in lighthouse_b200/ssz_schema.py) — no fork-specific oracle code involved."""
    from lighthouse_b200 import ssz_schema as S, tree_hash as T
    from lighthouse_b200.synthetic import beacon_state_deneb_ssz
    from tests import ssz_spec
    ssz = beacon_state_deneb_ssz(nv, seed=100 + nv, fork=fork, **kw)
    typ = S.BEACON_STATE_BY_FORK[fork]
    value = ssz_spec.deserialize(typ, ssz)
    assert S.serialize(typ, value) == ssz
    root, fields = T.beacon_state_root(ssz, fork, want_field_roots=True)
    want_fields = [ssz_spec.hash_tree_root(ft, value[name]) for name, ft in typ[1]]
    assert fields[:len(want_fields)] == want_fields, [i for i, (a, b) in enumerate(zip(fields, want_fields)) if a != b]
    assert root == ssz_spec.hash_tree_root(typ, value)
    if fork == "deneb":
        assert root == T.beacon_state_root_deneb(ssz)
    if fork == "electra" and nv == 37:               # pending_* lists at other lengths, incl. empty and one element
        for n_pending in ((0, 0, 0), (1, 1, 1), (4097, 2, 300)):
            ssz2 = beacon_state_deneb_ssz(nv, seed=7, fork=fork, n_pending=n_pending)
            assert T.beacon_state_root(ssz2, fork) == ssz_spec.hash_tree_root(typ, ssz_spec.deserialize(typ, ssz2)), n_pending
    # the wrong fork id must not silently produce a root of the same bytes' other interpretation
    other = {"altair": "deneb", "bellatrix": "capella", "capella": "deneb", "deneb": "capella", "electra": "deneb"}[fork]
    try:
        assert T.beacon_state_root(ssz, other) != root
    except Exception:
        pass                                          # rejected as malformed: also fine
