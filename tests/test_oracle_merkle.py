"""Pins the tree-hash oracle (oracle/ssz_sha256.c) against independent implementations and the reference's
own in-tree golden vectors (SURVEY.md §8c).  CPU only."""
import hashlib
import os
import struct

import numpy as np
import pytest

from tests import oracle_lib as O


def py_merkleize(chunks, depth):
    """independent hashlib restatement"""
    zero = [b"\0" * 32]
    for _ in range(64):
        zero.append(hashlib.sha256(zero[-1] * 2).digest())
    nodes = [chunks[i:i + 32] for i in range(0, len(chunks), 32)]
    if not nodes:
        return zero[depth]
    for lvl in range(depth):
        if len(nodes) % 2:
            nodes.append(zero[lvl])
        nodes = [hashlib.sha256(nodes[i] + nodes[i + 1]).digest() for i in range(0, len(nodes), 2)]
    return nodes[0]


def test_sha256_matches_hashlib_both_backends():
    rng = np.random.default_rng(0)
    for force_plain in (1, 0):
        O.L.orc_sha_backend(force_plain)
        for n in [0, 1, 31, 32, 55, 56, 63, 64, 65, 119, 120, 127, 128, 1000]:
            m = rng.integers(0, 256, n, dtype=np.uint8).tobytes()
            assert O.sha256(m) == hashlib.sha256(m).digest()
        d = rng.integers(0, 256, 64 * 100, dtype=np.uint8).tobytes()
        assert O.hash_pairs(d) == b"".join(hashlib.sha256(d[i:i + 64]).digest() for i in range(0, len(d), 64))


def test_zero_hashes():
    z = b"\0" * 32
    for d in range(0, 41):
        assert O.zero_hash(d) == z
        z = hashlib.sha256(z + z).digest()


@pytest.mark.parametrize("n,depth", [(0, 0), (0, 5), (1, 0), (1, 3), (2, 1), (3, 2), (5, 3), (5, 10), (8, 3),
                                     (9, 40), (1000, 10), (1025, 11), (4097, 20)])
def test_merkleize_matches_python(n, depth):
    rng = np.random.default_rng(n * 131 + depth)
    c = rng.integers(0, 256, 32 * n, dtype=np.uint8).tobytes()
    assert O.merkleize(c, depth) == py_merkleize(c, depth)


@pytest.mark.parametrize("net", ["sepolia", "gnosis", "mainnet"])
def test_genesis_validators_root_golden(net):
    meta = O.golden_json("genesis_validators.json")[net]
    ssz = O.golden_validators(net)
    lo = meta.get("stored_from", 0)
    assert len(ssz) == 121 * (meta["n_validators"] - lo)
    for threads in (1, 4):
        O.set_threads(threads)
        if lo:   # validators [lo, n) stored, with the root of the subtree over [0, lo)
            d = lo.bit_length() - 1
            node = O.hash_pairs(bytes.fromhex(meta["left_subtree_root"]) + O.merkleize(O.validator_roots(ssz), d))
            for lvl in range(d + 1, 40):
                node = O.hash_pairs(node + O.zero_hash(lvl))
            root = O.mix_in_length(node, meta["n_validators"])
        else:
            root = O.validators_root(ssz)
        assert root.hex() == meta["genesis_validators_root"]
    O.set_threads(1)


def test_deposit_roots_golden():
    """deposit_message_root / deposit_data_root of validator_manager/test_vectors
    (create_validators.rs:754-768): containers {pubkey, wc, amount} and {pubkey, wc, amount, signature}."""
    for d in O.golden_json("deposit_data.json"):
        pk = bytes.fromhex(d["pubkey"]); wc = bytes.fromhex(d["withdrawal_credentials"])
        amount = struct.pack("<Q", d["amount"]) + b"\0" * 24
        sig = bytes.fromhex(d["signature"])
        pk_root = O.merkleize_bytes(pk, 1)
        sig_root = O.merkleize_bytes(sig, 2)
        assert O.merkleize(pk_root + wc + amount, 2).hex() == d["deposit_message_root"]
        assert O.merkleize(pk_root + wc + amount + sig_root, 2).hex() == d["deposit_data_root"]


def test_merkle_tree_proof_roundtrip():
    rng = np.random.default_rng(7)
    for depth, n in [(0, 1), (1, 1), (3, 5), (5, 32), (12, 6), (32, 9)]:
        leaves = [rng.integers(0, 256, 32, dtype=np.uint8).tobytes() for _ in range(n)]
        for idx in {0, n - 1, min(n, (1 << depth) - 1)}:
            root, br = O.merkle_tree_proof(leaves, depth, idx)
            assert root == py_merkleize(b"".join(leaves), depth)
            leaf = leaves[idx] if idx < n else b"\0" * 32
            assert O.merkle_root_from_branch(leaf, br, depth, idx) == root


def test_beacon_state_field_rules():
    """Full-state oracle vs an independent python composition on a small synthetic Deneb state."""
    from lighthouse_b200.synthetic import beacon_state_deneb_ssz
    ssz = beacon_state_deneb_ssz(300, seed=3, n_hist_roots=5, n_votes=7, n_summaries=3)
    root, fr = O.beacon_state_root_deneb(ssz)
    assert root == py_merkleize(b"".join(fr), 5)
    # spot-check a few fields independently
    assert fr[5] == py_merkleize(ssz[176:176 + 8192 * 32], 13)
    o_val, o_bal = struct.unpack_from("<II", ssz, 524552)
    o_pp, = struct.unpack_from("<I", ssz, 2687248)
    vr = O.validator_roots(ssz[o_val:o_bal])
    assert fr[11] == hashlib.sha256(py_merkleize(vr, 40) + struct.pack("<Q", 300) + b"\0" * 24).digest()
    bal = ssz[o_bal:o_pp]
    bal += b"\0" * (-len(bal) % 32)
    assert fr[12] == hashlib.sha256(py_merkleize(bal, 38) + struct.pack("<Q", 300) + b"\0" * 24).digest()
    assert fr[17] == bytes([ssz[2687256]]) + b"\0" * 31


@pytest.mark.parametrize("kw", [dict(n_validators=37, seed=3, n_hist_roots=5, n_votes=7, n_summaries=3),
                                dict(n_validators=0, all_default=True),
                                dict(n_validators=1, seed=4, n_hist_roots=0, n_votes=0, n_summaries=0, extra_data_len=0),
                                dict(n_validators=1000, seed=9, extra_data_len=32)])
def test_state_oracle_matches_generic_spec_merkleization(kw):
    """Second, independent pin of the hand-unrolled BeaconStateDeneb oracle (the reference's own pin, EF ssz_static,
    is not on disk): decode the synthetic SSZ with the generic decoder of tests/ssz_spec.py, re-serialise (must be
    identical), and compare the root and ALL 28 field roots with the from-spec hashlib merkleization driven by the
    type descriptors in lighthouse_b200/ssz_schema.py (beacon_state.rs:339-490)."""
    from lighthouse_b200 import ssz_schema as S
    from lighthouse_b200.synthetic import beacon_state_deneb_ssz
    from tests import ssz_spec
    ssz = beacon_state_deneb_ssz(**kw)
    value = ssz_spec.deserialize(S.BeaconStateDeneb, ssz)
    assert S.serialize(S.BeaconStateDeneb, value) == ssz
    want_fields = [ssz_spec.hash_tree_root(ft, value[name]) for name, ft in S.BeaconStateDeneb[1]]
    root, fields = O.beacon_state_root_deneb(ssz)
    assert list(fields) == want_fields
    assert root == ssz_spec.hash_tree_root(S.BeaconStateDeneb, value)
