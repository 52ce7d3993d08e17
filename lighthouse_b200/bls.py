"""Host-side mirror of Lighthouse's `crypto/bls` surface for the B200 backend.

Names, argument meaning and error behaviour follow /root/reference/crypto/bls/src:
    PublicKey            generic_public_key.rs:46-102      (deserialize rejects infinity / bad points)
    Signature            generic_signature.rs:49-150       (all-zero bytes = "empty" signature, point None)
    AggregateSignature   generic_aggregate_signature.rs:60-235
    SecretKey / Keypair  generic_secret_key.rs, keypair.rs
    SignatureSet         generic_signature_set.rs:61-121
    verify_signature_sets  impls/blst.rs:37-119
Point types hold canonical bytes (like impls/fake_crypto.rs); every group operation is executed by the CUDA
library through the C ABI (include/lhb200.h).  There is no CPU arithmetic in this module.
"""
import ctypes as C

import numpy as np

from . import _ffi
from ._ffi import lib, check, buf

PUBLIC_KEY_BYTES_LEN = 48
PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN = 96
SIGNATURE_BYTES_LEN = 96
SECRET_KEY_BYTES_LEN = 32
INFINITY_PUBLIC_KEY = bytes([0xC0]) + bytes(47)
INFINITY_SIGNATURE = bytes([0xC0]) + bytes(95)
NONE_SIGNATURE = bytes(96)  # EMPTY_SIGNATURE_SERIALIZATION
CURVE_ORDER = 0x73EDA753299D7D483339D80809A1D80553BDA402FFFE5BFEFFFFFFFF00000001


class Error(Exception):
    """bls::Error (crypto/bls/src/lib.rs:49-62)"""


class InvalidByteLength(Error):
    pass


class InvalidInfinityPublicKey(Error):
    pass


class BlstError(Error):
    """decode / subgroup failure reported by the backend"""


class InvalidSecretKeyLength(Error):
    pass


class InvalidZeroSecretKey(Error):
    pass


def decompress_validate_pubkeys(compressed: bytes):
    """Batch PublicKey::deserialize: n x 48 bytes -> (n x 96 uncompressed bytes, status uint8[n])."""
    n = len(compressed) // 48
    out = np.zeros(n * 96, dtype=np.uint8)
    st = np.zeros(n, dtype=np.uint8)
    p, k = buf(compressed)
    check(lib.lhb200_g1_decompress_validate(p, n, out.ctypes.data, st.ctypes.data), "lhb200_g1_decompress_validate")
    return out.tobytes(), st


class PublicKey:
    """A validated G1 public key; keeps both serialisations (48-byte compressed, 96-byte uncompressed)."""
    __slots__ = ("compressed", "uncompressed")

    def __init__(self, compressed: bytes, uncompressed: bytes):
        self.compressed, self.uncompressed = compressed, uncompressed

    @classmethod
    def deserialize(cls, b: bytes) -> "PublicKey":
        if len(b) != PUBLIC_KEY_BYTES_LEN:
            raise InvalidByteLength(f"got {len(b)}, expected {PUBLIC_KEY_BYTES_LEN}")
        if b == INFINITY_PUBLIC_KEY:  # generic_public_key.rs:87-88
            raise InvalidInfinityPublicKey()
        unc, st = decompress_validate_pubkeys(b)
        if st[0] == 1:
            raise InvalidInfinityPublicKey()
        if st[0] != 0:
            raise BlstError(f"key_validate status {int(st[0])}")
        return cls(bytes(b), unc)

    @classmethod
    def deserialize_uncompressed(cls, b: bytes) -> "PublicKey":
        """TPublicKey::deserialize_uncompressed (blst.rs:142-150; generic_public_key.rs:97-102): encoding + curve
        check, no subgroup check; infinity is rejected like `deserialize`."""
        if len(b) != PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN:
            raise InvalidByteLength(f"got {len(b)}, expected {PUBLIC_KEY_UNCOMPRESSED_BYTES_LEN}")
        c48 = np.zeros(48, dtype=np.uint8)
        st = np.zeros(1, dtype=np.uint8)
        p, k = buf(b)
        check(lib.lhb200_g1_deserialize_uncompressed(p, 1, c48.ctypes.data, st.ctypes.data),
              "lhb200_g1_deserialize_uncompressed")
        if st[0] == 1:
            raise InvalidInfinityPublicKey()
        if st[0] != 0:
            raise BlstError("bad uncompressed G1 encoding")
        return cls(c48.tobytes(), bytes(b))

    def serialize(self) -> bytes:
        return self.compressed

    def serialize_uncompressed(self) -> bytes:
        return self.uncompressed

    def __eq__(self, o):
        return isinstance(o, PublicKey) and self.compressed == o.compressed

    def __hash__(self):
        return hash(self.compressed)


class Signature:
    """G2 signature; `point is None` for the empty signature (all-zero serialisation)."""
    __slots__ = ("bytes_", "is_empty")

    def __init__(self, b: bytes):
        self.bytes_ = bytes(b)
        self.is_empty = self.bytes_ == NONE_SIGNATURE

    @classmethod
    def empty(cls):
        return cls(NONE_SIGNATURE)

    @classmethod
    def infinity(cls):
        return cls(INFINITY_SIGNATURE)

    @classmethod
    def deserialize(cls, b: bytes) -> "Signature":
        if len(b) != SIGNATURE_BYTES_LEN:
            raise InvalidByteLength(f"got {len(b)}, expected {SIGNATURE_BYTES_LEN}")
        if bytes(b) == NONE_SIGNATURE:
            return cls(b)
        out = C.create_string_buffer(192)
        st = C.create_string_buffer(1)
        p, k = buf(b)
        check(lib.lhb200_g2_decompress(p, 1, out, st), "lhb200_g2_decompress")
        if st.raw[0] == 2:
            raise BlstError("bad G2 encoding")
        return cls(b)

    def serialize(self) -> bytes:
        return self.bytes_

    def is_infinity(self) -> bool:
        return self.bytes_ == INFINITY_SIGNATURE

    def verify(self, pubkey: PublicKey, msg: bytes) -> bool:
        """GenericSignature::verify (generic_signature.rs:140): single-key verify, group-checks the signature."""
        return SignatureSet.single_pubkey(self, pubkey, msg).verify()


def aggregate_signatures(sigs96: bytes) -> bytes:
    """Sum of n compressed signatures (lhb200_g2_aggregate; TAggregateSignature::add_assign, blst.rs:230-237)."""
    n = len(sigs96) // 96
    out = C.create_string_buffer(96)
    p, k = buf(sigs96 if n else b"\0")
    rc = lib.lhb200_g2_aggregate(p, n, out)
    if rc == _ffi.EDECODE:
        raise BlstError("bad G2 encoding")
    check(rc, "lhb200_g2_aggregate")
    return out.raw


class AggregatePublicKey:
    """GenericAggregatePublicKey (generic_aggregate_public_key.rs:9-15, impls/blst.rs:160-184)."""
    __slots__ = ("pk",)

    def __init__(self, pk: PublicKey):
        self.pk = pk

    @classmethod
    def aggregate(cls, pubkeys) -> "AggregatePublicKey":
        pubkeys = list(pubkeys)
        if not pubkeys:
            raise BlstError("aggregate of no keys")   # blst: BLST_AGGR_TYPE_MISMATCH
        o48, o96 = C.create_string_buffer(48), C.create_string_buffer(96)
        p, k = buf(b"".join(x.serialize_uncompressed() for x in pubkeys))
        rc = lib.lhb200_g1_aggregate(p, len(pubkeys), o48, o96)
        if rc == _ffi.EDECODE:
            raise BlstError("bad G1 key")
        check(rc, "lhb200_g1_aggregate")
        return cls(PublicKey(o48.raw, o96.raw))

    def to_public_key(self) -> PublicKey:
        return self.pk


class AggregateSignature(Signature):
    """GenericAggregateSignature (generic_aggregate_signature.rs:60-235): the point is kept as its canonical bytes;
    `add_assign*` and every verification run on the device."""

    @classmethod
    def deserialize(cls, b: bytes) -> "AggregateSignature":
        s = Signature.deserialize(b)
        return cls(s.bytes_)

    def add_assign(self, other: Signature):
        """generic_aggregate_signature.rs:124-136: an empty `other` is ignored; an empty `self` starts from infinity."""
        if other.is_empty:
            return
        base = INFINITY_SIGNATURE if self.is_empty else self.bytes_
        self.bytes_ = aggregate_signatures(base + other.bytes_)
        self.is_empty = False

    def add_assign_aggregate(self, other: "AggregateSignature"):
        self.add_assign(other)

    @classmethod
    def aggregate(cls, signatures) -> "AggregateSignature":
        """All signatures in one device pass (what repeated add_assign computes)."""
        agg = cls.infinity()
        sigs = [s.bytes_ for s in signatures if not s.is_empty]
        if sigs:
            agg.bytes_ = aggregate_signatures(b"".join(sigs))
        return agg

    def aggregate_verify(self, msgs, pubkeys) -> bool:
        """generic_aggregate_signature.rs:213-222 -> blst.rs:263-273."""
        msgs, pubkeys = list(msgs), list(pubkeys)
        if not msgs or len(msgs) != len(pubkeys) or self.is_empty:
            return False
        ok = C.create_string_buffer(1)
        ps, k1 = buf(self.bytes_)
        pm, k2 = buf(b"".join(msgs))
        pp, k3 = buf(b"".join(k.serialize_uncompressed() for k in pubkeys))
        check(lib.lhb200_aggregate_verify(ps, pm, pp, len(msgs), ok), "lhb200_aggregate_verify")
        return ok.raw[0] == 1

    def fast_aggregate_verify(self, msg: bytes, pubkeys) -> bool:
        """generic_aggregate_signature.rs:187-196: empty key list -> False."""
        if not pubkeys:
            return False
        return SignatureSet.multiple_pubkeys(self, list(pubkeys), msg).verify()

    def eth_fast_aggregate_verify(self, msg: bytes, pubkeys) -> bool:
        """generic_aggregate_signature.rs:200-210: no keys + infinity signature -> True."""
        if not pubkeys and self.is_infinity():
            return True
        return self.fast_aggregate_verify(msg, pubkeys)


class SecretKey:
    __slots__ = ("be32",)

    def __init__(self, be32: bytes):
        self.be32 = be32

    @classmethod
    def deserialize(cls, b: bytes) -> "SecretKey":
        if len(b) != SECRET_KEY_BYTES_LEN:
            raise InvalidSecretKeyLength(f"got {len(b)}, expected {SECRET_KEY_BYTES_LEN}")
        v = int.from_bytes(b, "big")
        if v == 0:
            raise InvalidZeroSecretKey()
        if v >= CURVE_ORDER:
            raise BlstError("secret key >= r")
        return cls(bytes(b))

    def serialize(self) -> bytes:
        return self.be32

    def public_key(self) -> PublicKey:
        pk48, pk96 = sk_to_pk(self.be32)
        return PublicKey(pk48, pk96)

    def sign(self, msg: bytes) -> Signature:
        return Signature(sign(self.be32, msg))


class Keypair:
    def __init__(self, sk: SecretKey):
        self.sk = sk
        self.pk = sk.public_key()


def sk_to_pk(sks: bytes):
    """n x 32-byte big-endian scalars -> (n x 48 compressed, n x 96 uncompressed)."""
    n = len(sks) // 32
    o48 = np.zeros(n * 48, dtype=np.uint8)
    o96 = np.zeros(n * 96, dtype=np.uint8)
    p, k = buf(sks)
    check(lib.lhb200_sk_to_pk(p, n, o48.ctypes.data, o96.ctypes.data), "lhb200_sk_to_pk")
    return o48.tobytes(), o96.tobytes()


def sign(sks: bytes, msgs: bytes) -> bytes:
    n = len(sks) // 32
    assert len(msgs) == 32 * n
    o = np.zeros(n * 96, dtype=np.uint8)
    p, k = buf(sks)
    q, k2 = buf(msgs)
    check(lib.lhb200_sign(p, q, n, o.ctypes.data), "lhb200_sign")
    return o.tobytes()


class SignatureSet:
    """GenericSignatureSet {signature, signing_keys, message} (generic_signature_set.rs:61-121)."""
    __slots__ = ("signature", "signing_keys", "message")

    def __init__(self, signature, signing_keys, message: bytes):
        assert len(message) == 32
        self.signature, self.signing_keys, self.message = signature, signing_keys, message

    @classmethod
    def single_pubkey(cls, signature, signing_key, message):
        return cls(signature, [signing_key], message)

    @classmethod
    def multiple_pubkeys(cls, signature, signing_keys, message):
        return cls(signature, list(signing_keys), message)

    def verify(self) -> bool:
        """:111 — fast_aggregate_verify semantics for one set."""
        return verify_signature_sets([self])


def flatten_signature_sets(sets):
    """SoA buffers for the C ABI: (sigs n*96, msgs n*32, pks K*96, offsets uint32[n+1])."""
    sigs = b"".join(s.signature.serialize() for s in sets)
    msgs = b"".join(s.message for s in sets)
    offs = np.zeros(len(sets) + 1, dtype=np.uint32)
    parts = []
    for i, s in enumerate(sets):
        offs[i + 1] = offs[i] + len(s.signing_keys)
        parts.extend(k.serialize_uncompressed() for k in s.signing_keys)
    return sigs, msgs, b"".join(parts), offs


def verify_signature_sets_raw(sigs, msgs, pks, offsets, rands=None, want_status=False):
    n = len(offsets) - 1
    ok = C.create_string_buffer(1)
    st = np.zeros(max(n, 1), dtype=np.uint8)
    offs = np.ascontiguousarray(offsets, dtype=np.uint32)
    r = None if rands is None else np.ascontiguousarray(rands, dtype=np.uint64)
    ps, k1 = buf(sigs if len(sigs) else b"\0")
    pm, k2 = buf(msgs if len(msgs) else b"\0")
    pp, k3 = buf(pks if len(pks) else b"\0")
    check(lib.lhb200_verify_signature_sets(ps, pm, pp, offs.ctypes.data, None if r is None else r.ctypes.data, n, ok,
                                           st.ctypes.data), "lhb200_verify_signature_sets")
    res = ok.raw[0] == 1
    return (res, st[:n]) if want_status else res


def verify_signature_sets(sets, rands=None) -> bool:
    """bls::verify_signature_sets (impls/blst.rs:37-119).  Empty iterator -> False."""
    sets = list(sets)
    if not sets:
        return False
    sigs, msgs, pks, offs = flatten_signature_sets(sets)
    return verify_signature_sets_raw(sigs, msgs, pks, offs, rands)


def verify_signature_set_groups_raw(sigs, msgs, pks, offsets, group_offsets, rands=None, want_status=False):
    """lhb200_verify_signature_set_groups: SoA buffers as verify_signature_sets_raw plus group_offsets (uint32[G+1], CSR
    over the sets).  -> list of G bools, each what verify_signature_sets_raw returns for that group's sets alone
    (and the per-set statuses with want_status)."""
    n = len(offsets) - 1
    goffs = np.ascontiguousarray(group_offsets, dtype=np.uint32)
    g = len(goffs) - 1
    if g < 0:
        raise ValueError("group_offsets needs at least one entry")
    ok = np.zeros(max(g, 1), dtype=np.uint8)
    st = np.zeros(max(n, 1), dtype=np.uint8)
    offs = np.ascontiguousarray(offsets, dtype=np.uint32)
    r = None if rands is None else np.ascontiguousarray(rands, dtype=np.uint64)
    ps, k1 = buf(sigs if len(sigs) else b"\0")
    pm, k2 = buf(msgs if len(msgs) else b"\0")
    pp, k3 = buf(pks if len(pks) else b"\0")
    check(lib.lhb200_verify_signature_set_groups(ps, pm, pp, offs.ctypes.data, None if r is None else r.ctypes.data, n,
                                                 goffs.ctypes.data, g, ok.ctypes.data, st.ctypes.data),
          "lhb200_verify_signature_set_groups")
    res = [bool(v) for v in ok[:g]]
    return (res, st[:n]) if want_status else res


def verify_signature_set_groups(groups, rands=None) -> list:
    """Many independent verify_signature_sets calls in one device pass: groups is a list of lists of SignatureSet;
    element g of the result is verify_signature_sets(groups[g]) (an empty group -> False)."""
    groups = [list(gr) for gr in groups]
    sets = [s for gr in groups for s in gr]
    goffs = np.zeros(len(groups) + 1, dtype=np.uint32)
    goffs[1:] = np.cumsum([len(gr) for gr in groups], dtype=np.uint64) if groups else []
    sigs, msgs, pks, offs = flatten_signature_sets(sets)
    return verify_signature_set_groups_raw(sigs, msgs, pks, offs, goffs, rands)


class ParallelSignatureSets:
    """state_processing::per_block_processing::block_signature_verifier::ParallelSignatureSets
    (block_signature_verifier.rs:84-96, :392-418): the sets of 1..N blocks are accumulated, then verified by ONE
    verify_signature_sets call (what BlockSignatureVerifier::verify and the chain-segment import do)."""

    def __init__(self, sets=None):
        self.sets = list(sets) if sets else []

    def push(self, signature_set: SignatureSet):
        self.sets.append(signature_set)

    def extend(self, sets):
        self.sets.extend(sets)

    def __len__(self):
        return len(self.sets)

    def verify(self) -> bool:
        return verify_signature_sets(self.sets)


class PubkeyTable:
    """Device-resident validator pubkey table (mirror of ValidatorPubkeyCache, validator_pubkey_cache.rs)."""

    def __init__(self, capacity):
        self._h = C.c_void_p()
        check(lib.lhb200_pubkey_table_create(capacity, C.byref(self._h)), "lhb200_pubkey_table_create")

    def append(self, pks96: bytes):
        p, k = buf(pks96)
        n = (len(pks96) if isinstance(pks96, (bytes, bytearray)) else k.nbytes) // 96
        check(lib.lhb200_pubkey_table_append(self._h, p, n), "lhb200_pubkey_table_append")

    def __len__(self):
        return int(lib.lhb200_pubkey_table_len(self._h))

    def destroy(self):
        if self._h:
            lib.lhb200_pubkey_table_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


class Batch:
    """Staged verify (lhb200_bls_batch_*): device-resident inputs, enqueue on a stream, read the verdict."""

    def __init__(self, max_sets, max_keys):
        self._h = C.c_void_p()
        check(lib.lhb200_bls_batch_create(max_sets, max_keys, C.byref(self._h)), "lhb200_bls_batch_create")
        self.n = 0

    def upload(self, sigs, msgs, pks, offsets, rands=None):
        offs = np.ascontiguousarray(offsets, dtype=np.uint32)
        self.n = len(offs) - 1
        r = None if rands is None else np.ascontiguousarray(rands, dtype=np.uint64)
        ps, k1 = buf(sigs); pm, k2 = buf(msgs); pp, k3 = buf(pks)
        check(lib.lhb200_bls_batch_upload(self._h, ps, pm, pp, offs.ctypes.data, None if r is None else r.ctypes.data,
                                          self.n), "lhb200_bls_batch_upload")

    def upload_async(self, sigs, msgs, pks, offsets, rands=None, stream=None):
        """Streamed upload (lhb200_bls_batch_upload_async): key chunks overlap the kernels of the following enqueue().
        The buffers are kept alive on the object until the next upload."""
        offs = np.ascontiguousarray(offsets, dtype=np.uint32)
        self.n = len(offs) - 1
        r = None if rands is None else np.ascontiguousarray(rands, dtype=np.uint64)
        ps, k1 = buf(sigs); pm, k2 = buf(msgs); pp, k3 = buf(pks)
        self._keep = (k1, k2, k3, offs, r)
        check(lib.lhb200_bls_batch_upload_async(self._h, ps, pm, pp, offs.ctypes.data,
                                                None if r is None else r.ctypes.data, self.n, stream),
              "lhb200_bls_batch_upload_async")

    def upload_indexed(self, table, sigs, msgs, indices, offsets, rands=None):
        offs = np.ascontiguousarray(offsets, dtype=np.uint32)
        idx = np.ascontiguousarray(indices, dtype=np.uint32)
        self.n = len(offs) - 1
        r = None if rands is None else np.ascontiguousarray(rands, dtype=np.uint64)
        ps, k1 = buf(sigs); pm, k2 = buf(msgs)
        check(lib.lhb200_bls_batch_upload_indexed(self._h, table._h, ps, pm, idx.ctypes.data, offs.ctypes.data,
                                                  None if r is None else r.ctypes.data, self.n),
              "lhb200_bls_batch_upload_indexed")

    def set_device_inputs(self, d_sigs, d_msgs, d_pks, d_offsets, d_rands, n):
        self.n = n
        check(lib.lhb200_bls_batch_set_device_inputs(self._h, d_sigs, d_msgs, d_pks, d_offsets, d_rands, n),
              "lhb200_bls_batch_set_device_inputs")

    def enqueue(self, stream=None):
        check(lib.lhb200_bls_batch_verify_enqueue(self._h, stream), "lhb200_bls_batch_verify_enqueue")

    def result(self, stream=None, want_status=False):
        ok = C.create_string_buffer(1)
        st = np.zeros(max(self.n, 1), dtype=np.uint8)
        check(lib.lhb200_bls_batch_result(self._h, stream, ok, st.ctypes.data if want_status else None),
              "lhb200_bls_batch_result")
        return (ok.raw[0] == 1, st[: self.n]) if want_status else ok.raw[0] == 1

    def gt_bytes(self):
        out = C.create_string_buffer(576)
        check(lib.lhb200_bls_batch_gt(self._h, out), "lhb200_bls_batch_gt")
        return out.raw

    @property
    def launches(self):
        return lib.lhb200_bls_batch_launches(self._h)

    @property
    def dominant_kernel_ms(self):
        return float(lib.lhb200_bls_batch_dominant_kernel_ms(self._h))

    def destroy(self):
        if self._h:
            lib.lhb200_bls_batch_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def debug_stage(op, data: bytes, out_len: int):
    """lhb200_debug_bls test hook -> (rc, out bytes)"""
    out = C.create_string_buffer(out_len)
    rc = C.c_int32(0)
    p, k = buf(data)
    check(lib.lhb200_debug_bls(op, p, len(data), out, out_len, C.byref(rc)), "lhb200_debug_bls")
    return rc.value, out.raw
