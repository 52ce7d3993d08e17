"""ctypes binding of liblhb200.so (the C ABI in include/lhb200.h).

The CUDA library is the product: if it is missing this module raises at import (no CPU fallback,
no routing through oracle/).  The library is built in-tree by `__graft_entry__.build()` /
`make -C lighthouse_b200/csrc`.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("LHB200_LIB_PATH", os.path.join(_HERE, "liblhb200.so"))  # override: tuning experiments only

if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
        "(lighthouse_b200 has no CPU fallback)")

lib = C.CDLL(LIB_PATH)

OK, ENODEV, EINVAL, ECUDA, ENOMEM, EDECODE = 0, -1, -2, -3, -4, -5
u8p, u32p, u64p, vp = C.POINTER(C.c_uint8), C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.c_void_p


class Lhb200Error(RuntimeError):
    def __init__(self, code, where):
        self.code = code
        msg = lib.lhb200_last_error().decode(errors="replace")
        super().__init__(f"{where}: status {code}: {msg}")


def _sig(name, restype, *argtypes):
    f = getattr(lib, name)
    f.restype = restype
    f.argtypes = list(argtypes)
    return f


_sig("lhb200_init", C.c_int32, C.c_int32)
_sig("lhb200_shutdown", None)
_sig("lhb200_last_error", C.c_char_p)
_sig("lhb200_pinned_alloc", C.c_int32, C.POINTER(vp), C.c_uint64)
_sig("lhb200_pinned_free", C.c_int32, vp)
_sig("lhb200_launch_count", C.c_uint64)
_sig("lhb200_hash_pairs", C.c_int32, vp, vp, C.c_uint64)
_sig("lhb200_dev_hash_pairs", C.c_int32, vp, vp, C.c_uint64, vp)
_sig("lhb200_merkleize", C.c_int32, vp, C.c_uint64, C.c_uint32, vp)
_sig("lhb200_dev_merkleize", C.c_int32, vp, C.c_uint64, C.c_uint32, vp, vp)
_sig("lhb200_mix_in_length", C.c_int32, vp, C.c_uint64, vp)
_sig("lhb200_zero_hash", C.c_int32, C.c_uint32, vp)
_sig("lhb200_validators_root", C.c_int32, vp, C.c_uint64, vp)
_sig("lhb200_validator_roots", C.c_int32, vp, C.c_uint64, vp)
_sig("lhb200_beacon_state_root_deneb", C.c_int32, vp, C.c_uint64, vp, vp)
_sig("lhb200_state_stage_deneb", C.c_int32, vp, C.c_uint64, C.POINTER(vp))
_sig("lhb200_state_root", C.c_int32, vp, vp, vp)
_sig("lhb200_state_root_enqueue", C.c_int32, vp, vp, C.POINTER(vp))
_sig("lhb200_state_release", C.c_int32, vp)
_sig("lhb200_state_hash_units", C.c_uint64, vp)
_sig("lhb200_merkle_tree_proof", C.c_int32, vp, C.c_uint64, C.c_uint32, C.c_uint64, vp, vp)
_sig("lhb200_verify_merkle_proofs", C.c_int32, vp, vp, C.c_uint32, vp, vp, C.c_uint64, vp)


def check(code, where):
    if code != OK:
        raise Lhb200Error(code, where)


_inited = None


def init(device=0):
    """lhb200_init; raises Lhb200Error(ENODEV) when no B200 is usable."""
    global _inited
    if _inited == device:
        return
    check(lib.lhb200_init(device), "lhb200_init")
    _inited = device


def buf(b):
    """bytes / bytearray / numpy array -> (c_void_p, keepalive)"""
    if isinstance(b, (bytes, bytearray)):
        arr = (C.c_uint8 * max(len(b), 1)).from_buffer_copy(b if len(b) else b"\0")
        return C.cast(arr, vp), arr
    import numpy as np
    a = np.ascontiguousarray(b)
    return C.c_void_p(a.ctypes.data), a

# ---- BLS path
_sig("lhb200_verify_signature_sets", C.c_int32, vp, vp, vp, vp, vp, C.c_uint32, vp, vp)
_sig("lhb200_verify_signature_set_groups", C.c_int32, vp, vp, vp, vp, vp, C.c_uint32, vp, C.c_uint32, vp, vp)
_sig("lhb200_bls_batch_create", C.c_int32, C.c_uint32, C.c_uint64, C.POINTER(vp))
_sig("lhb200_bls_batch_destroy", C.c_int32, vp)
_sig("lhb200_bls_batch_upload", C.c_int32, vp, vp, vp, vp, vp, vp, C.c_uint32)
_sig("lhb200_bls_batch_set_device_inputs", C.c_int32, vp, vp, vp, vp, vp, vp, C.c_uint32)
_sig("lhb200_bls_batch_verify_enqueue", C.c_int32, vp, vp)
_sig("lhb200_bls_batch_result", C.c_int32, vp, vp, vp, vp)
_sig("lhb200_bls_batch_gt", C.c_int32, vp, vp)
_sig("lhb200_bls_batch_launches", C.c_uint64, vp)
_sig("lhb200_sk_to_pk", C.c_int32, vp, C.c_uint32, vp, vp)
_sig("lhb200_sign", C.c_int32, vp, vp, C.c_uint32, vp)
_sig("lhb200_g1_decompress_validate", C.c_int32, vp, C.c_uint32, vp, vp)
_sig("lhb200_g2_decompress", C.c_int32, vp, C.c_uint32, vp, vp)
_sig("lhb200_debug_bls", C.c_int32, C.c_int32, vp, C.c_uint32, vp, C.c_uint32, C.POINTER(C.c_int32))
_sig("lhb200_bls_batch_dominant_kernel_ms", C.c_float, vp)
_sig("lhb200_state_dominant_kernel_ms", C.c_float, vp)
_sig("lhb200_pubkey_table_create", C.c_int32, C.c_uint64, C.POINTER(vp))
_sig("lhb200_pubkey_table_destroy", C.c_int32, vp)
_sig("lhb200_pubkey_table_append", C.c_int32, vp, vp, C.c_uint64)
_sig("lhb200_pubkey_table_len", C.c_uint64, vp)
_sig("lhb200_bls_batch_upload_indexed", C.c_int32, vp, vp, vp, vp, vp, vp, vp, C.c_uint32)
_sig("lhb200_state_stage_deneb_shard", C.c_int32, vp, C.c_uint64, C.c_uint32, C.c_uint32, C.POINTER(vp))
_sig("lhb200_state_shard_roots", C.c_int32, vp, vp, C.POINTER(C.c_uint32))
_sig("lhb200_state_combine", C.c_int32, vp, vp, vp)
_sig("lhb200_state_patch", C.c_int32, vp, C.c_uint64, vp, C.c_uint64)
_sig("lhb200_shuffle_list", C.c_int32, vp, C.c_uint64, C.c_uint8, vp, C.c_int32, vp)
_sig("lhb200_beacon_block_root_deneb", C.c_int32, vp, C.c_uint64, vp, vp)
_sig("lhb200_beacon_block_roots_deneb", C.c_int32, vp, vp, C.c_uint32, vp, vp)
_sig("lhb200_bls_batch_upload_async", C.c_int32, vp, vp, vp, vp, vp, vp, C.c_uint32, vp)
_sig("lhb200_state_enable_incremental", C.c_int32, vp)
_sig("lhb200_state_last_root_hashes", C.c_uint64, vp)
_sig("lhb200_state_patch_batch", C.c_int32, vp, vp, vp, vp, C.c_uint32)
_sig("lhb200_blinded_beacon_block_roots_deneb", C.c_int32, vp, vp, C.c_uint32, vp, vp)
_sig("lhb200_beacon_block_roots", C.c_int32, vp, vp, C.c_uint32, C.c_int32, C.c_int32, vp, vp)
_sig("lhb200_debug_rand_scalars", C.c_int32, vp, C.c_uint32)
_sig("lhb200_g2_aggregate", C.c_int32, vp, C.c_uint32, vp)
_sig("lhb200_g1_aggregate", C.c_int32, vp, C.c_uint32, vp, vp)
_sig("lhb200_g1_deserialize_uncompressed", C.c_int32, vp, C.c_uint32, vp, vp)
_sig("lhb200_aggregate_verify", C.c_int32, vp, vp, vp, C.c_uint32, vp)
_sig("lhb200_comm_unique_id", C.c_int32, vp)
_sig("lhb200_comm_init", C.c_int32, C.c_int32, C.c_int32, vp)
_sig("lhb200_comm_destroy", C.c_int32)
_sig("lhb200_comm_info", C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32))
_sig("lhb200_verify_signature_sets_collective", C.c_int32, vp, vp, vp, vp, vp, C.c_uint32, vp)
_sig("lhb200_bls_batch_allreduce_verdict", C.c_int32, vp, vp)
_sig("lhb200_state_root_sharded", C.c_int32, vp, vp)
_sig("lhb200_beacon_state_root", C.c_int32, vp, C.c_uint64, C.c_int32, vp, vp)
_sig("lhb200_state_stage", C.c_int32, vp, C.c_uint64, C.c_int32, C.POINTER(vp))
