"""ctypes access to oracle/liboracle.so — TEST INFRASTRUCTURE ONLY (never imported by lighthouse_b200/)."""
import ctypes as C
import json
import lzma
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_SO = os.path.join(ROOT, "oracle", "liboracle.so")
if not os.path.exists(_SO):
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle")])
L = C.CDLL(_SO)
L.orc_hw_threads.restype = C.c_int
GOLDEN = os.path.join(ROOT, "tests", "golden")


def _out32():
    return C.create_string_buffer(32)


def sha256(m: bytes) -> bytes:
    o = _out32(); L.orc_sha256(m, C.c_uint64(len(m)), o); return o.raw


def hash32_concat(a, b):
    o = _out32(); L.orc_hash32_concat(a, b, o); return o.raw


def hash_pairs(data: bytes) -> bytes:
    n = len(data) // 64
    o = C.create_string_buffer(max(32 * n, 1)); L.orc_hash_pairs(data, o, C.c_uint64(n)); return o.raw[:32 * n]


def zero_hash(d):
    o = _out32(); L.orc_zero_hash(C.c_uint32(d), o); return o.raw


def merkleize(chunks: bytes, depth: int) -> bytes:
    o = _out32(); L.orc_merkleize(chunks, C.c_uint64(len(chunks) // 32), C.c_uint32(depth), o); return o.raw


def merkleize_bytes(data: bytes, depth: int) -> bytes:
    o = _out32(); L.orc_merkleize_bytes(data, C.c_uint64(len(data)), C.c_uint32(depth), o); return o.raw


def mix_in_length(root, n):
    o = _out32(); L.orc_mix_in_length(root, C.c_uint64(n), o); return o.raw


def validator_roots(ssz: bytes) -> bytes:
    n = len(ssz) // 121
    o = C.create_string_buffer(max(32 * n, 1)); L.orc_validator_roots(ssz, C.c_uint64(n), o); return o.raw[:32 * n]


def validators_root(ssz: bytes) -> bytes:
    o = _out32(); L.orc_validators_root(ssz, C.c_uint64(len(ssz) // 121), o); return o.raw


def beacon_state_root_deneb(ssz: bytes):
    o = _out32(); fr = C.create_string_buffer(28 * 32)
    rc = L.orc_beacon_state_root_deneb(ssz, C.c_uint64(len(ssz)), o, fr)
    if rc:
        raise ValueError(f"oracle rejected state: {rc}")
    return o.raw, [fr.raw[32 * i:32 * i + 32] for i in range(28)]


def merkle_tree_proof(leaves, depth, index):
    root = _out32(); br = C.create_string_buffer(max(32 * depth, 1))
    L.orc_merkle_tree_proof(b"".join(leaves), C.c_uint64(len(leaves)), C.c_uint32(depth), C.c_uint64(index), root, br)
    return root.raw, [br.raw[32 * i:32 * i + 32] for i in range(depth)]


def merkle_root_from_branch(leaf, branch, depth, index):
    o = _out32()
    L.orc_merkle_root_from_branch(leaf, b"".join(branch), C.c_uint32(depth), C.c_uint64(index), o)
    return o.raw


def set_threads(n):
    L.orc_set_threads(C.c_int(n))


def hw_threads():
    return L.orc_hw_threads()


def golden_json(name):
    return json.load(open(os.path.join(GOLDEN, name)))


def golden_validators(net):
    """The stored SSZ validators of a genesis state: the whole list, or the list from index `stored_from` on when
    genesis_validators.json gives one (mainnet)."""
    return lzma.open(os.path.join(GOLDEN, f"genesis_validators_{net}.bin.xz")).read()


# ---- BLS C oracle (oracle/bls12_381.c)
import numpy as _np


def bls_verify_signature_sets(sigs, msgs, pks, offsets, rands, want_gt=False, want_muls=False, want_status=False):
    n = len(offsets) - 1
    offs = _np.ascontiguousarray(offsets, dtype=_np.uint32)
    r = _np.ascontiguousarray(rands, dtype=_np.uint64)
    st = _np.zeros(max(n, 1), dtype=_np.uint8)
    gt = C.create_string_buffer(576)
    muls = C.c_uint64(0)
    L.orc_verify_signature_sets.restype = C.c_int
    ok = L.orc_verify_signature_sets(sigs, msgs, pks, C.c_void_p(offs.ctypes.data), C.c_void_p(r.ctypes.data),
                                     C.c_uint32(n), C.c_void_p(st.ctypes.data), gt, C.byref(muls))
    out = [bool(ok)]
    if want_gt:
        out.append(gt.raw)
    if want_muls:
        out.append(muls.value)
    if want_status:
        out.append(st[:n])
    return out[0] if len(out) == 1 else tuple(out)


def bls_hash_to_g2(msg):
    o = C.create_string_buffer(96); L.orc_hash_to_g2(msg, o); return o.raw


def bls_sk_to_pk(sk_be32):
    o = C.create_string_buffer(96); L.orc_sk_to_pk(sk_be32, o); return o.raw


def bls_sign(sk_be32, msg):
    o = C.create_string_buffer(96); L.orc_sign(sk_be32, msg, o); return o.raw


def shuffle_list(values, rounds, seed, forwards):
    a = _np.ascontiguousarray(values, dtype=_np.uint64).copy()
    rc = L.orc_shuffle_list(C.c_void_p(a.ctypes.data), C.c_uint64(len(a)), C.c_uint8(rounds), seed, C.c_int(1 if forwards else 0))
    return None if rc else a.tolist()


def compute_shuffled_index(index, n, seed, rounds):
    L.orc_compute_shuffled_index.restype = C.c_int64
    v = L.orc_compute_shuffled_index(C.c_uint64(index), C.c_uint64(n), seed, C.c_uint8(rounds))
    return None if v < 0 else int(v)


def beacon_block_root_deneb(ssz):
    """-> (root, body_root) or None when the oracle rejects the SSZ."""
    out, body = (C.c_uint8 * 32)(), (C.c_uint8 * 32)()
    rc = L.orc_beacon_block_root_deneb(bytes(ssz), C.c_uint64(len(ssz)), out, body)
    return None if rc else (bytes(out), bytes(body))


def blinded_beacon_block_root_deneb(ssz):
    out, body = (C.c_uint8 * 32)(), (C.c_uint8 * 32)()
    rc = L.orc_blinded_beacon_block_root_deneb(bytes(ssz), C.c_uint64(len(ssz)), out, body)
    return None if rc else (bytes(out), bytes(body))
