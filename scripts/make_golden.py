#!/usr/bin/env python3
"""Extract the reference's own in-tree golden vectors into tests/golden/.

    python scripts/make_golden.py <sigp/lighthouse v5.3.0 checkout>

Sources (all under that checkout):
  common/eth2_network_config/built_in_network_configs/{mainnet,sepolia,gnosis}/genesis.ssz.zip
      phase0 genesis BeaconState; bytes 8..40 = genesis_validators_root = hash_tree_root(validators)
      (checked by common/eth2_network_config/src/lib.rs:227-233)
  validator_manager/test_vectors/vectors/*/validator_keys/deposit_data-*.json
      22 (pubkey, signature, deposit_message_root, deposit_data_root) entries, asserted valid by
      validator_manager/src/create_validators.rs:749-768
  common/eth2_interop_keypairs/specs/keygen_10_validators.yaml  (sk -> pk, tests/generation.rs:6-64)
Every fixture stays under 1 MB.  The mainnet list (21 063 validators, 1.6 MB compressed) is therefore stored from
validator 2^14 on, with the root of the subtree over the first 2^14 validators; the tests rebuild
genesis_validators_root from the two.
"""
import glob, hashlib, io, json, lzma, os, struct, sys, zipfile
import yaml

REF = sys.argv[1]
OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden")
os.makedirs(OUT, exist_ok=True)

# phase0 BeaconState fixed part: offset of the `validators` u32 offset (SURVEY §8c)
VAL_OFF_POS = 8 + 32 + 8 + 16 + 112 + 2 * 8192 * 32 + 4 + 72 + 4 + 8
MAINNET_STORED_FROM = 1 << 14


def merkle_root(chunks):
    """root over a power-of-two number of 32-byte chunks"""
    while len(chunks) > 1:
        chunks = [hashlib.sha256(chunks[i] + chunks[i + 1]).digest() for i in range(0, len(chunks), 2)]
    return chunks[0]


def validator_root(v):
    """hash_tree_root of one 121-byte SSZ Validator"""
    u64 = lambda o: v[o:o + 8] + bytes(24)
    pubkey = hashlib.sha256(v[0:32] + v[32:48] + bytes(16)).digest()
    return merkle_root([pubkey, v[48:80], u64(80), v[88:89] + bytes(31), u64(89), u64(97), u64(105), u64(113)])


meta = {}
for net in ("mainnet", "sepolia", "gnosis"):
    z = zipfile.ZipFile(f"{REF}/common/eth2_network_config/built_in_network_configs/{net}/genesis.ssz.zip")
    state = z.read(z.namelist()[0])
    o_val, o_bal = struct.unpack_from("<II", state, VAL_OFF_POS)
    vals = state[o_val:o_bal]
    assert len(vals) % 121 == 0
    meta[net] = {"n_validators": len(vals) // 121, "genesis_validators_root": state[8:40].hex()}
    if net == "mainnet":
        lo = MAINNET_STORED_FROM
        assert lo < len(vals) // 121 <= 2 * lo
        meta[net] |= {"stored_from": lo, "left_subtree_root": merkle_root(
            [validator_root(vals[121 * i:121 * i + 121]) for i in range(lo)]).hex()}
        vals = vals[121 * lo:]
    with lzma.open(os.path.join(OUT, f"genesis_validators_{net}.bin.xz"), "wb", preset=9) as f:
        f.write(vals)
json.dump(meta, open(os.path.join(OUT, "genesis_validators.json"), "w"), indent=1)

deps = []
for p in sorted(glob.glob(f"{REF}/validator_manager/test_vectors/vectors/*/validator_keys/deposit_data-*.json")):
    for d in json.load(open(p)):
        deps.append({k: d[k] for k in ("pubkey", "withdrawal_credentials", "amount", "signature",
                                        "deposit_message_root", "deposit_data_root", "fork_version")}
                    | {"source": os.path.relpath(p, REF)})
json.dump(deps, open(os.path.join(OUT, "deposit_data.json"), "w"), indent=1)

kp = yaml.safe_load(open(f"{REF}/common/eth2_interop_keypairs/specs/keygen_10_validators.yaml"))
json.dump(kp, open(os.path.join(OUT, "interop_keypairs.json"), "w"), indent=1)
print({k: v["n_validators"] for k, v in meta.items()}, len(deps), "deposits", len(kp), "keypairs")
