"""lhb200_verify_signature_set_groups on the device: one verdict per group of SignatureSets.  Every expected verdict is
the CPU oracle's orc_verify_signature_sets run on that group's sets alone, with the same blinding scalars."""
import hashlib
import json
import os
import subprocess
import sys
import threading
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import bls_ref as B
from tests import oracle_lib as O

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def bls(gpu):
    from lighthouse_b200 import bls as m
    return m


def batch(n_sets, keys_per_set, seed):
    from lighthouse_b200.synthetic import attestation_batch
    ab = attestation_batch(n_sets, keys_per_set=keys_per_set, n_validators=1024, seed=seed)
    return bytearray(ab.sigs), bytearray(ab.msgs), bytearray(ab.pks), np.asarray(ab.offsets, dtype=np.uint32)


def rands_for(n, seed):
    return np.random.default_rng(seed).integers(1, 2 ** 63, size=n, dtype=np.uint64)


def offsets(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint32)


def oracle_verdicts(sigs, msgs, pks, offs, goffs, rands):
    """orc_verify_signature_sets per group (an empty group: False), groups spread over the CPU cores."""
    sigs, msgs, pks = bytes(sigs), bytes(msgs), bytes(pks)
    offs = np.asarray(offs, dtype=np.int64)

    def one(g):
        lo, hi = int(goffs[g]), int(goffs[g + 1])
        if lo == hi:
            return False
        k0, k1 = int(offs[lo]), int(offs[hi])
        return bool(O.bls_verify_signature_sets(sigs[96 * lo:96 * hi], msgs[32 * lo:32 * hi], pks[96 * k0:96 * k1] or b"\0",
                                                offs[lo:hi + 1] - k0, rands[lo:hi]))

    saved = O.L.orc_num_threads()
    O.set_threads(1)   # one oracle thread per group, the groups in parallel
    try:
        with ThreadPoolExecutor(max(1, os.cpu_count() or 1)) as ex:
            return list(ex.map(one, range(len(goffs) - 1)))
    finally:
        O.set_threads(saved)


def flip_msg(msgs, i):
    msgs[32 * i] ^= 1


def test_per_set_verdicts_cfg0_shape(bls):
    """64 one-set groups of 128 keys (BASELINE configs[0] shape): a wrong message at set 0, a valid signature by another
    key at set 17, one wrong key out of 128 at set 63 -> exactly those three groups fail."""
    sigs, msgs, pks, offs = batch(64, 128, seed=3)
    flip_msg(msgs, 0)
    sigs[96 * 17:96 * 18] = bls.sign((777).to_bytes(32, "big"), bytes(msgs[32 * 17:32 * 18]))
    k = int(offs[63]) + 5
    pks[96 * k:96 * k + 96] = B.g1_uncompressed(B.sk_to_pk(987654321))
    goffs = np.arange(65, dtype=np.uint32)
    r = rands_for(64, 1)
    got, st = bls.verify_signature_set_groups_raw(bytes(sigs), bytes(msgs), bytes(pks), offs, goffs, r, want_status=True)
    assert [g for g in range(64) if not got[g]] == [0, 17, 63]
    assert not st.any()
    assert got == oracle_verdicts(sigs, msgs, pks, offs, goffs, r)


def test_aggregate_shape_groups_of_three(bls):
    """21 groups of 3 sets (an aggregate's selection proof, aggregator signature and attestation): one corrupted set
    fails its own group only."""
    sigs, msgs, pks, offs = batch(63, 16, seed=5)
    flip_msg(msgs, 3 * 7 + 1)
    goffs = offsets([3] * 21)
    r = rands_for(63, 2)
    got = bls.verify_signature_set_groups_raw(bytes(sigs), bytes(msgs), bytes(pks), offs, goffs, r)
    assert got == [g != 7 for g in range(21)]
    assert got == oracle_verdicts(sigs, msgs, pks, offs, goffs, r)


def _non_subgroup_g2():
    x = (3, 1)
    while True:
        y = B.f2_sqrt(B.f2_add(B.f2_mul(B.f2_sqr(x), x), B.B2))
        if y:
            return (x, y)
        x = (x[0] + 1, 1)


def _set(sk, msg, n_keys=1):
    """(sig96, msg32, [pk96]) with n_keys signers sk, sk+1, ..."""
    sks = [sk + i for i in range(n_keys)]
    return B.g2_compress(B.sign(sum(sks) % B.R, msg)), msg, [B.g1_uncompressed(B.sk_to_pk(s)) for s in sks]


def test_appendix_c_cases_each_in_its_own_group(bls):
    """Empty (all-zero) signature, infinity signature, no keys, aggregate key at infinity, undecodable signature and a
    signature outside G2, each inside its own group between valid ones: those groups fail, the others pass, and the
    per-set statuses are what lhb200_verify_signature_sets reports for the same sets."""
    m = [hashlib.sha256(b"appc%d" % i).digest() for i in range(16)]
    good = [_set(100 + 10 * i, m[i], n_keys=1 + i % 3) for i in range(8)]
    sig0, _, keys0 = good[0]
    pk5 = B.g1_uncompressed(B.sk_to_pk(5))
    undecodable = bytes([sig0[0] & 0x7F]) + sig0[1:]                         # compression flag cleared
    cases = [
        [good[0]],
        [(bytes(96), m[8], keys0)],                                          # empty signature -> status 1
        [good[1], (B.g2_compress(None), m[9], keys0)],                       # infinity signature
        [(sig0, m[10], [])],                                                 # no keys -> status 4
        [(sig0, m[11], [pk5, B.g1_uncompressed(B.g1_neg(B.sk_to_pk(5)))])],  # aggregate key at infinity -> 5
        [good[2], (undecodable, m[12], keys0)],                              # undecodable -> 2
        [(B.g2_compress(_non_subgroup_g2()), m[13], keys0)],                 # outside G2 -> 3
        [good[3], good[4], good[5]],
    ]
    flat = [s for grp in cases for s in grp]
    sigs = b"".join(s for s, _, _ in flat)
    msgs = b"".join(mm for _, mm, _ in flat)
    pks = b"".join(k for _, _, ks in flat for k in ks)
    offs = offsets([len(ks) for _, _, ks in flat])
    goffs = offsets([len(g) for g in cases])
    r = rands_for(len(flat), 3)
    got, st = bls.verify_signature_set_groups_raw(sigs, msgs, pks, offs, goffs, r, want_status=True)
    assert got == [True, False, False, False, False, False, False, True]
    assert got == oracle_verdicts(sigs, msgs, pks, offs, goffs, r)
    ok_plain, st_plain = bls.verify_signature_sets_raw(sigs, msgs, pks, offs, r, want_status=True)
    assert not ok_plain
    assert list(st) == list(st_plain)
    assert list(st) == [0, 1, 0, 0, 4, 5, 0, 2, 3, 0, 0, 0]


def test_empty_groups_and_malformed_offsets(bls):
    from lighthouse_b200._ffi import Lhb200Error, EINVAL
    sigs, msgs, pks, offs = batch(6, 4, seed=7)
    sigs, msgs, pks = bytes(sigs), bytes(msgs), bytes(pks)
    r = rands_for(6, 4)
    goffs = np.array([0, 2, 2, 5, 5, 6], dtype=np.uint32)                    # two empty groups
    assert bls.verify_signature_set_groups_raw(sigs, msgs, pks, offs, goffs, r) == [True, False, True, False, True]
    # more groups than sets, all but a few empty
    goffs = np.array([0] * 5 + [1, 1, 6] + [6] * 300, dtype=np.uint32)
    got = bls.verify_signature_set_groups_raw(sigs, msgs, pks, offs, goffs, r)
    assert len(got) == len(goffs) - 1 and [g for g in range(len(got)) if got[g]] == [4, 6]
    # no sets at all: every group empty; no groups at all
    assert bls.verify_signature_set_groups_raw(b"", b"", b"", np.zeros(1), np.zeros(4), None) == [False] * 3
    assert bls.verify_signature_set_groups_raw(b"", b"", b"", np.zeros(1), np.zeros(1), None) == []
    assert bls.verify_signature_set_groups([]) == []
    assert bls.verify_signature_set_groups([[], []]) == [False, False]
    for bad in ([1, 3, 6], [0, 4, 3, 6], [0, 2, 5], [0, 2, 7], [0]):
        with pytest.raises(Lhb200Error) as e:
            bls.verify_signature_set_groups_raw(sigs, msgs, pks, offs, np.array(bad, dtype=np.uint32), r)
        assert e.value.code == EINVAL, bad


def test_single_group_agrees_with_plain_call(bls):
    """n_groups == 1 takes the single-verdict path: same verdict and statuses as lhb200_verify_signature_sets on valid
    and invalid batches (both sides of the selection: the grouped kernels run for any other group count)."""
    sigs, msgs, pks, offs = batch(40, 8, seed=9)
    r = rands_for(40, 5)
    one = np.array([0, 40], dtype=np.uint32)
    for corrupt in (None, 11):
        m = bytearray(msgs)
        if corrupt is not None:
            flip_msg(m, corrupt)
        got, st = bls.verify_signature_set_groups_raw(bytes(sigs), bytes(m), bytes(pks), offs, one, r, want_status=True)
        plain, st_plain = bls.verify_signature_sets_raw(bytes(sigs), bytes(m), bytes(pks), offs, r, want_status=True)
        assert got == [plain] == [corrupt is None]
        assert list(st) == list(st_plain)
        two = bls.verify_signature_set_groups_raw(bytes(sigs), bytes(m), bytes(pks), offs, np.array([0, 20, 40]), r)
        assert two == [corrupt is None or corrupt >= 20, corrupt is None or corrupt < 20]


def test_random_group_sizes_across_the_latency_crossover(bls):
    """Groups of 1 ... 40 sets over ~1 000 sets (above the 888-set latency-mode crossover of the G2 stages), scattered
    corruptions of every kind (message, signature swap, key)."""
    rng = np.random.default_rng(11)
    sizes = []
    while sum(sizes) < 1000:
        sizes.append(int(rng.integers(1, 41)))
    n = sum(sizes)
    sigs, msgs, pks, offs = batch(n, 4, seed=13)
    victims = sorted(rng.choice(n, size=12, replace=False).tolist())
    for j, v in enumerate(victims):
        if j % 3 == 0:
            flip_msg(msgs, v)
        elif j % 3 == 1:
            w = (v + 1) % n
            sigs[96 * v:96 * v + 96], sigs[96 * w:96 * w + 96] = sigs[96 * w:96 * w + 96], sigs[96 * v:96 * v + 96]
        else:
            k = int(offs[v])
            pks[96 * k:96 * k + 96] = B.g1_uncompressed(B.sk_to_pk(424242 + v))
    goffs = offsets(sizes)
    r = rands_for(n, 6)
    got = bls.verify_signature_set_groups_raw(bytes(sigs), bytes(msgs), bytes(pks), offs, goffs, r)
    want = oracle_verdicts(sigs, msgs, pks, offs, goffs, r)
    assert got == want
    assert 0 < want.count(False) <= 24


def test_ten_thousand_per_set_verdicts(bls):
    """10 000 one-set groups (20 000 Miller pairs: several waves of the pair kernel, 10 000 final exponentiations) with
    scattered bad sets."""
    n = 10000
    sigs, msgs, pks, offs = batch(n, 1, seed=17)
    rng = np.random.default_rng(12)
    victims = sorted(rng.choice(n, size=40, replace=False).tolist())
    for v in victims:
        flip_msg(msgs, v)
    goffs = np.arange(n + 1, dtype=np.uint32)
    r = rands_for(n, 7)
    got = bls.verify_signature_set_groups_raw(bytes(sigs), bytes(msgs), bytes(pks), offs, goffs, r)
    assert [i for i in range(n) if not got[i]] == victims
    assert got == oracle_verdicts(sigs, msgs, pks, offs, goffs, r)


def test_library_drawn_scalars(bls):
    """rands = NULL: the library draws the blinding scalars; the verdicts do not depend on them."""
    sigs, msgs, pks, offs = batch(30, 3, seed=19)
    flip_msg(msgs, 4)
    flip_msg(msgs, 29)
    goffs = offsets([5, 1, 9, 10, 5])
    got = bls.verify_signature_set_groups_raw(bytes(sigs), bytes(msgs), bytes(pks), offs, goffs, None)
    assert got == [False, True, True, True, False]
    assert got == oracle_verdicts(sigs, msgs, pks, offs, goffs, rands_for(30, 8))


_MODE_PROBE = r"""
import json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import lighthouse_b200
from lighthouse_b200 import bls
from lighthouse_b200.synthetic import attestation_batch
lighthouse_b200.init(0)
ab = attestation_batch(48, keys_per_set=8, n_validators=1024, seed=23)
msgs = bytearray(ab.msgs); msgs[32 * 5] ^= 1
sigs = bytearray(ab.sigs); sigs[96 * 30:96 * 31] = bytes(96)
goffs = np.array([0, 1, 4, 10, 10, 29, 30, 31, 48], dtype=np.uint32)
r = np.arange(1, 49, dtype=np.uint64) * np.uint64(0x9E3779B97F4A7C15)
got, st = bls.verify_signature_set_groups_raw(bytes(sigs), bytes(msgs), ab.pks, ab.offsets, goffs, r, want_status=True)
per_set, _ = bls.verify_signature_set_groups_raw(bytes(sigs), bytes(msgs), ab.pks, ab.offsets, np.arange(49), r, want_status=True)
print(json.dumps({"groups": got, "per_set": per_set, "status": [int(x) for x in st]}))
"""


def test_lane_per_set_g2_stages_agree(bls):
    """LHB_G2_WARP=0 (the lane-per-set k_sig_prepare / k_hash_to_g2 in place of the warp-per-item ones; read once per
    process, hence subprocesses): same group verdicts, per-set verdicts and statuses."""
    root = O.ROOT

    def run(extra):
        out = subprocess.run([sys.executable, "-c", _MODE_PROBE, root], env=dict(os.environ, **extra), capture_output=True,
                             text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-2000:]
        return json.loads(out.stdout.strip().splitlines()[-1])

    warp, lane = run({}), run({"LHB_G2_WARP": "0"})
    assert warp == lane
    assert warp["groups"] == [True, True, False, False, True, True, False, True]
    assert [i for i, v in enumerate(warp["per_set"]) if not v] == [5, 30]
    assert [i for i, v in enumerate(warp["status"]) if v] == [30]


def test_grouped_and_plain_calls_from_several_threads(bls):
    """Grouped and plain calls at once from eight threads (each borrows its own pooled handle and stream)."""
    sigs, msgs, pks, offs = batch(32, 8, seed=29)
    flip_msg(msgs, 6)
    sigs, msgs, pks = bytes(sigs), bytes(msgs), bytes(pks)
    r = rands_for(32, 9)
    per_set = np.arange(33, dtype=np.uint32)
    quads = offsets([4] * 8)
    want_per_set = [i != 6 for i in range(32)]
    want_quads = [g != 1 for g in range(8)]
    errors = []

    def worker(t):
        try:
            for it in range(4):
                if (t + it) % 3 == 0:
                    assert bls.verify_signature_sets_raw(sigs, msgs, pks, offs, r) is False
                elif (t + it) % 3 == 1:
                    assert bls.verify_signature_set_groups_raw(sigs, msgs, pks, offs, per_set, r) == want_per_set
                else:
                    assert bls.verify_signature_set_groups_raw(sigs, msgs, pks, offs, quads, r) == want_quads
        except Exception as e:   # noqa: BLE001 — reported below
            errors.append((t, repr(e)))

    threads = [threading.Thread(target=worker, args=(t,)) for t in range(8)]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert not errors, errors


def test_python_mirror_groups_of_signature_sets(bls):
    """bls.verify_signature_set_groups on lists of SignatureSet objects == verify_signature_sets per group."""
    def make(ids, msg, valid=True):
        sks = [1000 + i for i in ids]
        keys = []
        for s in sks:
            pk = B.sk_to_pk(s)
            keys.append(bls.PublicKey(B.g1_compress(pk), B.g1_uncompressed(pk)))
        sig = B.g2_compress(B.sign(sum(sks) % B.R, msg if valid else hashlib.sha256(msg).digest()))
        return bls.SignatureSet.multiple_pubkeys(bls.AggregateSignature(sig), keys, msg)

    m = [hashlib.sha256(b"py%d" % i).digest() for i in range(6)]
    groups = [[make([0], m[0])], [make([1, 2], m[1]), make([3], m[2])], [], [make([4], m[3], valid=False)],
              [make([5, 6, 7], m[4]), make([8], m[5], valid=False)]]
    got = bls.verify_signature_set_groups(groups)
    assert got == [True, True, False, False, False]
    assert got == [bls.verify_signature_sets(g) for g in groups]


def test_cpp_host_layer_grouped_call(gpu, tmp_path):
    """include/lhb200.hpp: bls::verify_signature_set_groups (tests/cpp/group_verify_test.cpp, built here against the
    library) on the 22 deposit vectors."""
    deps = O.golden_json("deposit_data.json")
    vec = tmp_path / "vectors.bin"
    with open(vec, "wb") as f:
        for d in deps:
            fv = bytes.fromhex(d["fork_version"])
            fdr = hashlib.sha256(fv + bytes(28) + bytes(32)).digest()
            root = hashlib.sha256(bytes.fromhex(d["deposit_message_root"]) + bytes([3, 0, 0, 0]) + fdr[:28]).digest()
            f.write(bytes.fromhex(d["pubkey"]) + root + bytes.fromhex(d["signature"]))
    exe = tmp_path / "group_verify_test"
    lib_dir = os.path.join(O.ROOT, "lighthouse_b200")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-I" + os.path.join(O.ROOT, "include"), "-o", str(exe),
                           os.path.join(O.ROOT, "tests", "cpp", "group_verify_test.cpp"), "-L" + lib_dir, "-llhb200",
                           "-Wl,-rpath," + lib_dir])
    r = subprocess.run([str(exe), str(vec)], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "OK 29 groups" in r.stdout
