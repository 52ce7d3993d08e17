"""CPU-only: the device pieces of the grouped verification (lhb200_verify_signature_set_groups) compiled for the host
(tests/hostsim/hostsim_groups.cpp) and run lane by lane — the segmented sum r sig (gw::sum_points over the chunk tables of
bls/groups.cuh) and the per-group fold + final exponentiation of k_final_groups_warp (fe::group_verdict) — checked
against the big-integer oracle."""
import ctypes as C
import os
import random
import subprocess

import numpy as np
import pytest

from oracle import bls_ref as B
from tests import oracle_lib as O

HS = os.path.join(O.ROOT, "tests", "hostsim")


class _Libs:
    """hs_pairing from the shared host simulation (tests/hostsim/libhostsim.so), the grouped pieces from
    tests/hostsim/hostsim_groups.cpp, built here into a temporary directory"""
    def __init__(self, base, groups):
        self.hs_pairing = base.hs_pairing
        self.hs_g2_sum_seg = groups.hs_g2_sum_seg
        self.hs_final_groups = groups.hs_final_groups


@pytest.fixture(scope="module")
def L(tmp_path_factory):
    subprocess.check_call(["make", "-C", HS, "-s"])
    base = C.CDLL(os.path.join(HS, "libhostsim.so"))
    so = str(tmp_path_factory.mktemp("hostsim_groups") / "libhostsim_groups.so")
    subprocess.check_call([os.environ.get("CXX", "g++"), "-O2", "-std=c++17", "-fPIC", "-fvisibility=hidden", "-shared",
                           "-o", so, os.path.join(HS, "hostsim_groups.cpp")])
    groups = C.CDLL(so)
    base.hs_pairing.argtypes = [C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.c_char_p]
    groups.hs_g2_sum_seg.argtypes = [C.c_char_p, C.c_int, C.c_void_p, C.c_int, C.c_char_p]
    groups.hs_final_groups.argtypes = [C.c_char_p, C.c_void_p, C.c_char_p, C.c_char_p, C.c_void_p, C.c_int, C.c_char_p,
                                       C.c_char_p]
    return _Libs(base, groups)


def f12_from(bs):
    v = [(int.from_bytes(bs[96 * i:96 * i + 48], "big"), int.from_bytes(bs[96 * i + 48:96 * i + 96], "big"))
         for i in range(6)]
    return ((v[0], v[1], v[2]), (v[3], v[4], v[5]))


def offsets(sizes):
    return np.concatenate([[0], np.cumsum(sizes)]).astype(np.uint32)


def test_group_fold_and_final_exponentiation_match_oracle(L):
    """Groups of 1, 2, 3 and 9 Miller values plus the group's (-g1, sum) value: verdict and exponentiated value (the cube
    of the oracle's GT element) per group.  The 3-value group carries a wrong sum, one group is flagged failed by a set
    status, one group is empty: both decided without an exponentiation."""
    rnd = random.Random(17)
    groups = []   # per group: [(a, k)] pairs (a G1, k G2) and the scalar of the group's sum
    for size, wrong in ((1, False), (2, False), (3, True), (9, False), (2, False), (0, False)):
        pairs = [(rnd.randrange(1, 1 << 32), rnd.randrange(1, 1 << 32)) for _ in range(size)]
        s = sum(a * k for a, k in pairs) % B.R or 12345   # (the empty group's value is never read)
        groups.append((pairs, (s + 1) % B.R if wrong else s))
    failed = 4

    def miller_bytes(p, q):
        out = C.create_string_buffer(576)
        assert L.hs_pairing(B.g1_uncompressed(p), B.g2_compress(q), 0, 0, out) == 0
        return out.raw

    neg_g1 = B.g1_neg(B.G1_GEN)
    vals, extras, want = [], [], []
    for gi, (pairs, s) in enumerate(groups):
        pts = [(B.g1_mul(B.G1_GEN, a), B.g2_mul(B.G2_GEN, k)) for a, k in pairs]
        vals += [miller_bytes(p, q) for p, q in pts]
        extras.append(miller_bytes(neg_g1, B.g2_mul(B.G2_GEN, s)))
        if gi == failed or not pairs:
            want.append((False, None))
            continue
        f = B.miller_loop(neg_g1, B.g2_mul(B.G2_GEN, s))
        for p, q in pts:
            f = B.f12_mul(f, B.miller_loop(p, q))
        g = B.final_exp(f)
        want.append((g == B.F12_ONE, B.f12_mul(B.f12_sqr(g), g)))
    sizes = [len(p) for p, _ in groups]
    goff = offsets(sizes)
    status = bytearray(int(goff[-1]))
    status[int(goff[failed]) + 1] = 3
    ok, gt = C.create_string_buffer(len(groups)), C.create_string_buffer(576 * len(groups))
    assert L.hs_final_groups(b"".join(vals), goff.ctypes.data, b"".join(extras), bytes(status), goff.ctypes.data,
                             len(groups), ok, gt) == 0
    assert [v for v, _ in want] == [True, True, False, True, False, False]
    for g, (verdict, cube) in enumerate(want):
        assert ok.raw[g] == int(verdict), g
        if cube is None:
            assert gt.raw[576 * g:576 * g + 576] == bytes(576), g
        else:
            assert f12_from(gt.raw[576 * g:576 * g + 576]) == cube, g


def test_segmented_g2_sum_matches_oracle(L):
    """Per-group sums r sig over the level tables of bls/groups.cuh (chunks of four that stop at every group boundary):
    ragged groups whose boundaries fall inside the chunks an unsegmented level would use, infinity points inside a group,
    a group of nothing but infinities, an empty group and groups of 9 and 17 points (two and three levels) == the
    oracle's g2_add chain per group.  One point per group needs no level at all."""
    rnd = random.Random(31)
    sizes = [1, 3, 0, 5, 2, 9, 1, 4, 17, 2]
    n = sum(sizes)
    pts = [B.g2_mul(B.G2_GEN, rnd.randrange(1, B.R)) for _ in range(n)]
    goff = offsets(sizes)
    pts[int(goff[3]) + 2] = None                      # infinity inside a group
    pts[int(goff[4])] = pts[int(goff[4]) + 1] = None  # a group of infinities only
    enc = b"".join(B.g2_compress(p) for p in pts)
    out = C.create_string_buffer(96 * len(sizes))
    levels = L.hs_g2_sum_seg(enc, n, goff.ctypes.data, len(sizes), out)
    assert levels == 3                                # 17 -> 5 -> 2 -> 1
    for g in range(len(sizes)):
        acc = None
        for p in pts[goff[g]:goff[g + 1]]:
            if p is not None:
                acc = B.g2_add(acc, p)
        assert out.raw[96 * g:96 * g + 96] == B.g2_compress(acc), g
    # per-set groups: no level, the points are their own sums
    goff1 = offsets([1] * 6)
    out1 = C.create_string_buffer(96 * 6)
    assert L.hs_g2_sum_seg(b"".join(B.g2_compress(p) for p in pts[:6]), 6, goff1.ctypes.data, 6, out1) == 0
    assert out1.raw == b"".join(B.g2_compress(p) for p in pts[:6])
