"""Grouped verification (lhb200_verify_signature_set_groups) against the per-item calls it replaces.

Rows (one JSON line each, host wall clock around calls that return after a device synchronise, warm-up first, every
measurement at least --seconds of back-to-back calls, each configuration measured in --rounds alternating rounds):
  per_set_64      64 one-set groups (1 key, one bad set): one grouped call | 64 single-set verify_signature_sets calls
  aggregate_21x3  21 groups of 3 sets (1, 1 and 128 keys; one bad set): one grouped call | 21 three-set calls
  per_set_1000 / per_set_10000   per-set verdicts of 1 000 / 10 000 one-key sets: grouped call | one plain batch call
  single_group_64 a valid 64-set batch of 128-key sets through both entry points, n_groups = 1
The card's name and power limit (nvidia-smi, read-only query) go on every line.
usage: python scripts/quick_group_verify_bench.py [--out profiles/r3_group_verify.jsonl] [--seconds 1.0] [--rounds 2]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import lighthouse_b200
from lighthouse_b200 import bls
from lighthouse_b200.synthetic import interop_pubkey_table, materialize_sets, sets_workload


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


def make(key_counts, seed, table):
    ab = materialize_sets(sets_workload(np.asarray(key_counts), table.shape[0], seed), table, bls.sign)
    return bytearray(ab.sigs), bytearray(ab.msgs), bytes(ab.pks), np.asarray(ab.offsets, dtype=np.uint32)


def timed(fn, seconds):
    """ms per call over >= `seconds` of back-to-back calls (after 3 warm-up calls)"""
    for _ in range(3):
        fn()
    times = []
    t_end = time.perf_counter() + seconds
    while time.perf_counter() < t_end or len(times) < 3:
        t0 = time.perf_counter()
        fn()
        times.append(time.perf_counter() - t0)
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "r3_group_verify.jsonl"))
    ap.add_argument("--seconds", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=2)
    a = ap.parse_args()
    lighthouse_b200.init(0)
    name, power = card()
    table = interop_pubkey_table(1024)
    rows = []

    def sets_slice(sigs, msgs, pks, offs, lo, hi):
        k0, k1 = int(offs[lo]), int(offs[hi])
        return bytes(sigs[96 * lo:96 * hi]), bytes(msgs[32 * lo:32 * hi]), pks[96 * k0:96 * k1], offs[lo:hi + 1] - k0

    def grouped(sigs, msgs, pks, offs, goffs, want):
        sigs, msgs = bytes(sigs), bytes(msgs)
        def f():
            assert bls.verify_signature_set_groups_raw(sigs, msgs, pks, offs, goffs) == want
        return f

    def loop(sigs, msgs, pks, offs, goffs, want):
        parts = [sets_slice(sigs, msgs, pks, offs, int(goffs[g]), int(goffs[g + 1])) for g in range(len(goffs) - 1)]
        def f():
            assert [bls.verify_signature_sets_raw(*p) for p in parts] == want
        return f

    def plain(sigs, msgs, pks, offs, want):
        sigs, msgs = bytes(sigs), bytes(msgs)
        def f():
            assert bls.verify_signature_sets_raw(sigs, msgs, pks, offs) == want
        return f

    configs = []
    # 64 unaggregated attestations (one key each), one bad
    s, m, p, o = make([1] * 64, 31, table)
    m[32 * 40] ^= 1
    g = np.arange(65, dtype=np.uint32)
    want = [i != 40 for i in range(64)]
    configs.append(("per_set_64", 64, 64, "1", [("grouped", grouped(s, m, p, o, g, want)),
                                                ("loop_of_single_set_calls", loop(s, m, p, o, g, want))]))
    # 21 aggregates of 3 sets (selection proof, aggregator signature: one key; the attestation: 128 keys), one bad
    s, m, p, o = make([1, 1, 128] * 21, 32, table)
    m[32 * (3 * 9 + 2)] ^= 1
    g = np.arange(0, 64, 3, dtype=np.uint32)
    want = [i != 9 for i in range(21)]
    configs.append(("aggregate_21x3", 63, 21, "1,1,128", [("grouped", grouped(s, m, p, o, g, want)),
                                                          ("loop_of_per_aggregate_calls", loop(s, m, p, o, g, want))]))
    for n in (1000, 10000):
        s, m, p, o = make([1] * n, 33 + n, table)
        bad = list(range(7, n, n // 10))
        for i in bad:
            m[32 * i] ^= 1
        g = np.arange(n + 1, dtype=np.uint32)
        want = [i not in bad for i in range(n)]
        configs.append((f"per_set_{n}", n, n, "1", [("grouped", grouped(s, m, p, o, g, want)),
                                                    ("plain_single_verdict_same_batch", plain(s, m, p, o, False))]))
    s, m, p, o = make([128] * 64, 34, table)
    g = np.array([0, 64], dtype=np.uint32)
    configs.append(("single_group_64", 64, 1, "128", [("grouped_n_groups_1", grouped(s, m, p, o, g, [True])),
                                                      ("plain", plain(s, m, p, o, True))]))
    with open(a.out, "w") as f:
        for row, n_sets, n_groups, keys, variants in configs:
            for r in range(a.rounds):
                for label, fn in variants:
                    t = timed(fn, a.seconds)
                    rec = {"row": row, "entry": label, "round": r, "n_sets": n_sets, "n_groups": n_groups,
                           "keys_per_set": keys, "calls": len(t), "ms_mean": 1e3 * statistics.fmean(t),
                           "ms_median": 1e3 * statistics.median(t), "ms_min": 1e3 * min(t), "gpu": name,
                           "power_limit": power}
                    print(json.dumps(rec), flush=True)
                    f.write(json.dumps(rec) + "\n")


if __name__ == "__main__":
    main()
